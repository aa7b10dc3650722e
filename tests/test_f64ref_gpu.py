"""Every fp32 fused kernel form against the float64 reference of tests/f64ref.py, pixel by pixel, within the error bound
its arithmetic allows.

Each case names the kernel form it means to hit and asserts it through last_launch(); the last test asserts that every form
of the list below was launched and checked.  Inputs are impulse lattices (isolated values of 128, 2R+2 apart, shifted
along the diagonal over the batch so that an impulse lands on every column and every row: every column residue, both sides
of each 128-column strip seam and of each row-band seam (64 rows for G2, 90 for G4), both pixels of a two-pixel pair, the
first and last R+1 rows and columns) followed by two dense noise frames.  On an impulse frame the exact basis value is 128
times a sum of at most four tap products, so a wrong tap, reflection, halo, seam or pair store is an O(1) relative error.

16-bit output planes, host-buffer, band and multi-GPU paths are tested bit for bit against the fp32 device launch elsewhere
(test_out16_gpu.py, test_u8_in_gpu.py, test_bands_gpu.py, test_multi_gpu.py), so checking the fp32 forms covers them."""
import json
import os

import numpy as np
import pytest
import torch

from cvsteer_b200 import capi
from cvsteer_b200 import filters as cb
from cvsteer_b200.batch import G2Batch, G4Batch, pyr_down
from tests import f64ref as R
from tests import util

pytestmark = pytest.mark.gpu

F32 = np.float32
DOM, SCALAR, MAP = capi.STEER_DOMINANT, capi.STEER_SCALAR, capi.STEER_MAP
SCALARS = (1.5707, 1.5709, -1.5707, -1.5709, 0.7)

# --------------------------------------------------------------------------------------------------------------------------
# The kernel forms (the table of forms and launch_form in march_launch.cuh / march_forms.cuh):
#   every static mask: /tma/imm-taps (default taps, TMA-eligible fp32), /tma (other taps at the default width), /ldg (an
#   fp32 frame the TMA cannot address), /tma-u8 and /ldg-u8 (8-bit frames);
#   /tma/imm-taps/2px where the mask has a two-pixel instantiation (M2, lines, steer5, M2 and lines at a scalar, M2 at a
#   map) and the output layout allows pair stores (even width);
#   the run-time-mask kernels (<dyn>) have no baked-tap form;
#   widths other than the family default take the two-kernel generic path (generic_w<width>).
# --------------------------------------------------------------------------------------------------------------------------
G2_KERNELS = {   # name: (mask, steering source, two-pixel form?)
    "M0": (capi.G2_MASK_STATE, DOM, False),
    "M1": (capi.G2_MASK_ORIENT, DOM, False),
    "M2": (capi.G2_MASK_FULL, DOM, True),
    "lines": (capi.G2_MASK_LINES, DOM, True),
    "steer5@scalar": (capi.G2_MASK_STEER5, SCALAR, True),
    "steer5@map": (capi.G2_MASK_STEER5, MAP, True),
    "M2@scalar": (capi.G2_MASK_FULL, SCALAR, True),
    "M2@map": (capi.G2_MASK_FULL, MAP, True),
    "lines@scalar": (capi.G2_MASK_LINES, SCALAR, True),
    "lines@map": (capi.G2_MASK_LINES, MAP, False),
    "dyn": (capi.G2_MASK_STATE | capi.G2_MASK_FULL | capi.G2_MASK_LINES, DOM, False),
}
G4_KERNELS = {
    "basis": (capi.G4_MASK_BASIS, DOM, False),
    "steer@map": (capi.G4_MASK_STEER, MAP, False),
    "steer@scalar": (capi.G4_MASK_STEER, SCALAR, False),
    "steer@theta_d": (capi.G4_MASK_STEER, DOM, False),
    "dyn": (capi.G4_MASK_BASIS | capi.G4_MASK_STEER | capi.bit(capi.G4_THETA) | capi.bit(capi.G4_STRENGTH), DOM, False),
}
LOADERS = ("tma/imm-taps/2px", "tma/imm-taps", "tma", "ldg", "tma-u8", "ldg-u8")


def _forms(fam, kernels):
    out = []
    for k, (_, _, px2) in kernels.items():
        for ld in LOADERS:
            if k == "dyn" and "imm-taps" in ld:
                continue
            if ld.endswith("2px") and not px2:
                continue
            out.append((fam, k, ld))
    return out


FORMS = _forms(2, G2_KERNELS) + _forms(4, G4_KERNELS)
EXPECTED = sorted({f"g{f}_march<{k}>/{ld}" for f, k, ld in FORMS} | {"generic_w3", "generic_w5"} |
                  {"class:g2 setup", "class:g2 steer@scalar", "class:g2 steer@map", "class:g2 steer@theta_d",
                   "class:computeMagnitudeAndPhase", "class:find*", "class:g4 setup", "class:g4 steer@scalar",
                   "class:g4 steer@map", "pyr_down"})
SEEN = set()

# frame geometry: G2 frames span two 64-row band seams, G4 frames two 90-row seams; both span two 128-column strip seams
ROWS = {2: 140, 4: 190}
OTHER_SPACING = {2: 0.7, 4: 0.55}


def lattice(rows, cols, period, k):
    img = np.zeros((rows, cols), F32)
    img[k % period::period, k % period::period] = 128.0
    return img


def frames_for(fam, cols, u8, seed=0):
    """(frames [n, rows, cols], impulse flags): one impulse lattice per diagonal shift, then two dense frames."""
    R_ = 4 if fam == 2 else 6
    period = 2 * R_ + 2
    rows = ROWS[fam]
    imp = [lattice(rows, cols, period, k) for k in range(period)]
    rng = np.random.default_rng(100 + fam + seed)
    if u8:
        dense = [rng.integers(0, 256, (rows, cols)).astype(F32) for _ in range(2)]
    else:
        dense = [rng.uniform(0, 255, (rows, cols)).astype(F32) for _ in range(2)]
    return np.stack(imp + dense), [True] * period + [False] * 2


_REF_CACHE = {}


def reference(F, frames, impulse, key):
    """(B, beta, orientation) over the batch: planes [nb, n, rows, cols]."""
    ck = (F.fam, F.width, F.spacing, key)
    if ck not in _REF_CACHE:
        Bs, betas = [], []
        for f, imp in zip(frames, impulse):
            B, S = R.basis(f, F)
            Bs.append(B)
            betas.append(R.basis_bound(S, F, impulse=imp))
        B = np.stack(Bs, axis=1)
        beta = np.stack(betas, axis=1)
        if len(_REF_CACHE) > 6:                  # keep host memory bounded: a batch reference is ~100 MB
            _REF_CACHE.clear()
        _REF_CACHE[ck] = (B, beta, R.orientation(B, beta, F))
    return _REF_CACHE[ck]


def device_frames(frames, loader):
    """The frames as a CUDA tensor laid out so that the dispatch takes `loader`."""
    n, rows, cols = frames.shape
    u8 = loader.endswith("u8")
    dt = torch.uint8 if u8 else torch.float32
    src = torch.from_numpy(frames.astype(np.uint8) if u8 else frames)
    if loader.startswith("ldg"):                 # one element past an aligned base: not 16-byte aligned
        base = torch.zeros((n, rows, cols + 1), dtype=dt, device="cuda")
        x = base[:, :, 1:]
    else:                                        # 16-byte aligned rows: pitch padded to a multiple of 16 bytes
        es = 1 if u8 else 4
        pitch = -(-cols * es // 16) * 16 // es
        base = torch.zeros((n, rows, pitch), dtype=dt, device="cuda")
        x = base[:, :, :cols]
    x.copy_(src.cuda())
    return x


def _angle(label, got, want_bound, period, dense):
    """Angle check; on the dense frames of the batch (index list `dense`) at most 1 % of the pixels may be undetermined."""
    R.check_angle(label, got, want_bound, period)
    if dense:
        b = want_bound[1][dense]
        assert (b > R.EXCLUDE_RAD).sum() <= 0.01 * b.size, f"{label}: {(b > R.EXCLUDE_RAD).sum()} of {b.size} px undetermined"


def check_planes(label, F, ref, got, src, angle, fast, dense=()):
    """Every plane in `got` against the reference: basis, orientation, steering at the kernel's own angle, magnitude, phase,
    find*.  Static kernels use the SFU forms (fast); the run-time-mask and generic kernels the accurate ones."""
    B, beta, ori = ref
    names = set(got)
    for q, n in enumerate(F.names):
        if n in names:
            R.check(f"{label} {n}", got[n], (B[q], beta[q]))
    for k in ("c1", "c2", "c3", "strength"):
        if k in names:
            R.check(f"{label} {k}", got[k], ori[k])
    if "theta" in names:
        _angle(f"{label} theta", got["theta"], ori["theta"], np.pi, dense)
    gk, hk = ("g2", "h2") if F.fam == 2 else ("g4", "h4")
    steered = names & {gk, hk, "magnitude", "phase", "edges", "lines_dark", "lines_bright"}
    if not (steered or "e" in names):
        return
    dth = 0.0
    if src == DOM:
        if "theta" in names:
            th = got["theta"].astype(np.float64)
        else:                                    # steered to a theta_d the launch does not store: the reference's, with its bound
            th, dth = ori["theta"][0], np.minimum(ori["theta"][1], np.pi / 2)
        eps = R.EPS_SINCOS_FAST if fast else R.EPS_SINCOS_STEER
    elif src == SCALAR:
        th = np.full(B.shape[1:], float(F32(angle)))
        eps = R.EPS_SINCOS_HOST
    else:
        th = angle.astype(np.float64)
        eps = R.sincos_eps_fast(th) if fast else R.EPS_SINCOS_STEER
    if "e" in names:
        R.check(f"{label} e", got["e"], R.energy_dominant(ori) if src == DOM else R.energy(ori, th, eps, dth))
    if not steered:
        return
    g, h = R.steer(B, beta, F, th, eps, dth)
    if gk in names:
        R.check(f"{label} {gk}", got[gk], g)
    if hk in names:
        R.check(f"{label} {hk}", got[hk], h)
    m, p = R.mag_phase(g, h)
    if "magnitude" in names:
        R.check(f"{label} magnitude", got["magnitude"], m)
    if "phase" in names:
        _angle(f"{label} phase", got["phase"], p, 2 * np.pi, dense)
    fd = R.find(m, p, R.EPS_SINCOS_FAST if fast else R.EPS_SINCOS_STEER)
    for k in ("edges", "lines_dark", "lines_bright"):
        if k in names:
            R.check(f"{label} {k}", got[k], fd[k])


def _run_form(fam, kname, loader, angle_span=np.pi):
    kernels = G2_KERNELS if fam == 2 else G4_KERNELS
    mask, src, _ = kernels[kname]
    cols = 264 if loader.endswith("2px") else 263
    u8 = loader.endswith("u8")
    spacing = OTHER_SPACING[fam] if loader == "tma" and kname != "dyn" else None
    frames, impulse = frames_for(fam, cols, u8)
    F = R.family(fam, None, spacing)
    ref = reference(F, frames, impulse, (cols, u8))
    Batch = G2Batch if fam == 2 else G4Batch
    b = Batch() if spacing is None else Batch(spacing=spacing)
    x = device_frames(frames, loader)
    angle, kw = None, {}
    if src == SCALAR:
        angle = SCALARS[LOADERS.index(loader) % len(SCALARS)]
        kw = dict(steer=SCALAR, theta=angle)
    elif src == MAP:
        angle = np.random.default_rng(7).uniform(-angle_span, angle_span, frames.shape).astype(F32)
        kw = dict(steer=MAP, theta_map=torch.from_numpy(angle).cuda())
    res = b.run(x, mask, **kw)
    name = b.last_launch()["kernel"]
    want = f"g{fam}_march<{kname}>/{loader}"
    assert name == want, (name, want)
    SEEN.add(name)
    got = {k: v.cpu().numpy() for k, v in res.items()}
    dense = [i for i, imp in enumerate(impulse) if not imp]
    check_planes(name, F, ref, got, src, angle, fast=kname != "dyn" and kname != "M0", dense=dense)
    return name


@pytest.mark.parametrize("fam,kname,loader", FORMS, ids=[f"g{f}-{k}-{ld}" for f, k, ld in FORMS])
def test_kernel_form_vs_f64(fam, kname, loader):
    _run_form(fam, kname, loader)


@pytest.mark.parametrize("fam,kname", [(2, "steer5@map"), (4, "steer@map")])
def test_sincos_beyond_pi(fam, kname):
    """Angle maps in [-8, 8]: __sincosf's argument reduction, against the families.cuh figure beyond pi."""
    _run_form(fam, kname, "tma/imm-taps", angle_span=8.0)


@pytest.mark.parametrize("fam,width", [(2, 3), (4, 5)])
def test_generic_width_vs_f64(fam, width):
    frames, impulse = frames_for(fam, 263, False)
    F = R.family(fam, width, 0.67 if fam == 2 else 0.5)
    ref = reference(F, frames, impulse, (263, False))
    b = G2Batch(width=width) if fam == 2 else G4Batch(width=width)
    x = torch.from_numpy(frames).cuda()
    mask = (capi.G2_MASK_STATE | capi.G2_MASK_FULL | capi.G2_MASK_LINES) if fam == 2 else G4_KERNELS["dyn"][0]
    res = b.run(x, mask)
    name = b.last_launch()["kernel"]
    assert name == f"generic_w{width}", name
    SEEN.add(name)
    check_planes(name, F, ref, {k: v.cpu().numpy() for k, v in res.items()}, DOM, None, fast=False, dense=[len(frames) - 1])
    tmap = np.random.default_rng(8).uniform(-np.pi, np.pi, frames.shape).astype(F32)
    steer_mask = capi.G2_MASK_STEER5 if fam == 2 else capi.G4_MASK_STEER
    res = b.run(x, steer_mask, steer=MAP, theta_map=torch.from_numpy(tmap).cuda())
    check_planes(name + "@map", F, ref, {k: v.cpu().numpy() for k, v in res.items()}, MAP, tmap, fast=False,
                 dense=[len(frames) - 1])


DENSE_SHAPES = [(72, 256), (130, 131), (91, 257), (200, 520), (5, 300), (1, 1), (3, 5), (7, 7)]


@pytest.mark.parametrize("shape", DENSE_SHAPES, ids=[f"{r}x{c}" for r, c in DENSE_SHAPES])
@pytest.mark.parametrize("u8", [False, True], ids=["f32", "u8"])
def test_dense_shapes_vs_f64(shape, u8):
    """Dense frames on shapes around the tiling edges; the smallest ones take the cooperative loader."""
    rng = np.random.default_rng(shape[0] * 1000 + shape[1])
    frames = (rng.integers(0, 256, (2,) + shape) if u8 else rng.uniform(0, 255, (2,) + shape)).astype(F32)
    x = torch.from_numpy(frames.astype(np.uint8) if u8 else frames).cuda()
    tmap = rng.uniform(-np.pi, np.pi, frames.shape).astype(F32)
    for fam, kname in ((2, "M2"), (2, "steer5@map"), (4, "basis"), (4, "steer@map")):
        F = R.family(fam)
        ref = reference(F, frames, [False, False], ("dense", shape, u8))
        mask, src, _ = (G2_KERNELS if fam == 2 else G4_KERNELS)[kname]
        b = G2Batch() if fam == 2 else G4Batch()
        kw = dict(steer=MAP, theta_map=torch.from_numpy(tmap).cuda()) if src == MAP else {}
        res = b.run(x, mask, **kw)
        name = b.last_launch()["kernel"]
        assert name.startswith(f"g{fam}_march<{kname}>/"), name
        SEEN.add(name)
        got = {k: v.cpu().numpy() for k, v in res.items()}
        dense = [0, 1] if frames[0].size >= 1000 else []    # a few pixels have no determined orientation
        check_planes(f"{name} {shape}", F, ref, got, src, tmap if src == MAP else None, fast=True, dense=dense)
        lvl = pyr_down(x.float() if u8 else x)
        SEEN.add("pyr_down")
        for i in range(2):
            R.check(f"pyr_down {shape}", lvl[i].cpu().numpy(), R.pyr_down(frames[i]))


def test_pyr_down_impulses():
    frames, _ = frames_for(2, 263, False)
    lvl = pyr_down(torch.from_numpy(frames).cuda()).cpu().numpy()
    SEEN.add("pyr_down")
    for i, f in enumerate(frames):
        R.check("pyr_down impulses", lvl[i], R.pyr_down(f))


@pytest.mark.parametrize("fam", [2, 4])
def test_full_hd_frame(fam):
    img = util.synth(1080 + fam, 1080, 1920)
    F = R.family(fam)
    ref = reference(F, img[None], [False], ("1080p",))
    kname = "M2" if fam == 2 else "steer@map"
    mask, src, _ = (G2_KERNELS if fam == 2 else G4_KERNELS)[kname]
    tmap = np.random.default_rng(9).uniform(-np.pi, np.pi, (1, 1080, 1920)).astype(F32)
    b = G2Batch() if fam == 2 else G4Batch()
    kw = dict(steer=MAP, theta_map=torch.from_numpy(tmap).cuda()) if src == MAP else {}
    res = b.run(torch.from_numpy(img[None]).cuda(), mask, **kw)
    name = b.last_launch()["kernel"]
    check_planes(f"{name} 1080p", F, ref, {k: v.cpu().numpy() for k, v in res.items()}, src, tmap, fast=True, dense=[0])


def test_class_api_vs_f64():
    """The class-API kernels: setup (the state planes), steer at a scalar, at a map and at the handle's own theta_d,
    computeMagnitudeAndPhase and find* on given planes, and G4 setup / steer."""
    frames, impulse = frames_for(2, 263, False)
    tmap = np.random.default_rng(10).uniform(-np.pi, np.pi, frames.shape[1:]).astype(F32)
    for i in (3, len(frames) - 1):               # one impulse lattice, one dense frame
        img = frames[i]
        F = R.family(2)
        ref = reference(F, img[None], [impulse[i]], ("class", i))
        f = cb.SteerableFiltersG2(img)
        got = {n: f.plane(capi.G2_PLANE_NAMES.index(n))[None] for n in capi.G2_PLANE_NAMES[:12]}
        check_planes("class g2 setup", F, ref, got, DOM, None, fast=False)
        SEEN.add("class:g2 setup")
        keys = ("g2", "h2", "e", "magnitude", "phase")
        for tag, arg, src, ang in (("steer@scalar", 0.7, SCALAR, 0.7), ("steer@map", tmap, MAP, tmap[None]),
                                   ("steer@theta_d", None, MAP, got["theta"])):
            out = f.steer(arg)
            check_planes(f"class g2 {tag}", F, ref, {k: v[None] for k, v in zip(keys, out)}, src, ang, fast=False)
            SEEN.add(f"class:g2 {tag}")
        g2, h2 = out[0], out[1]
        mag, ph = f.computeMagnitudeAndPhase(g2, h2)
        exact = (g2.astype(np.float64), np.zeros(g2.shape)), (h2.astype(np.float64), np.zeros(h2.shape))
        m, p = R.mag_phase(*exact)
        R.check("class computeMagnitudeAndPhase magnitude", mag, m)
        R.check_angle("class computeMagnitudeAndPhase phase", ph, p, 2 * np.pi)
        SEEN.add("class:computeMagnitudeAndPhase")
        fd = R.find((mag.astype(np.float64), np.zeros(mag.shape)), (ph.astype(np.float64), np.zeros(ph.shape)),
                    R.EPS_SINCOS_STEER)
        R.check("class findEdges", f.findEdges(mag, ph), fd["edges"])
        R.check("class findDarkLines", f.findDarkLines(mag, ph), fd["lines_dark"])
        R.check("class findBrightLines", f.findBrightLines(mag, ph), fd["lines_bright"])
        SEEN.add("class:find*")
    frames4, impulse4 = frames_for(4, 263, False)
    for i in (5, len(frames4) - 1):
        img = frames4[i]
        F = R.family(4)
        ref = reference(F, img[None], [impulse4[i]], ("class", i))
        f4 = cb.SteerableFiltersG4(img)
        got = {n: f4.plane(capi.G4_PLANE_NAMES.index(n))[None] for n in capi.G4_PLANE_NAMES[:11]}
        got["theta"] = f4.getDominantOrientationAngle()[None]
        got["strength"] = f4.getDominantOrientationStrength()[None]
        check_planes("class g4 setup", F, ref, got, DOM, None, fast=False)
        SEEN.add("class:g4 setup")
        keys = ("g4", "h4", "magnitude", "phase")
        out = f4.steer(0.3, with_phase=True)
        check_planes("class g4 steer@scalar", F, ref, {k: v[None] for k, v in zip(keys, out)}, SCALAR, 0.3, fast=False)
        SEEN.add("class:g4 steer@scalar")
        tm4 = np.random.default_rng(11).uniform(-np.pi, np.pi, img.shape).astype(F32)
        out = f4.steer(tm4, with_phase=True)
        check_planes("class g4 steer@map", F, ref, {k: v[None] for k, v in zip(keys, out)}, MAP, tm4[None], fast=False)
        SEEN.add("class:g4 steer@map")


def test_every_form_was_checked():
    """Runs last: every kernel form of the list was launched and checked in this session.  With CVS_F64_BOUNDS_JSON set to a
    file path, writes the per (kernel, quantity) maxima of err / bound there (profiles/r05_f64_bounds.json is one such run)."""
    missing = sorted(set(EXPECTED) - SEEN)
    summary = {}
    for r in util.RECORDS:
        if r["kind"] != "f64bound":
            continue
        s = summary.setdefault(r["name"], {"max_err_over_bound": 0.0, "excluded_px": 0, "px": 0})
        s["max_err_over_bound"] = max(s["max_err_over_bound"], r["err"])
        s["excluded_px"] += r.get("excluded", 0)
        s["px"] += r["n"]
    path = os.environ.get("CVS_F64_BOUNDS_JSON")
    if path:
        with open(path, "w") as f:
            json.dump({"gpu": torch.cuda.get_device_name(0), "forms_checked": sorted(SEEN),
                       "quantities": dict(sorted(summary.items()))}, f, indent=1)
    assert not missing, f"kernel forms never checked: {missing}"
