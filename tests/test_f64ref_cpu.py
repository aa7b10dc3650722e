"""The float64 reference and its per-pixel bounds (tests/f64ref.py), proven on the CPU: the reference matches cv2, correct
float32 arithmetic (the cv2 oracle, and a float32 emulation with another summation order) passes every check at every pixel,
and subtle defects of the kind a kernel could share across all its forms are rejected."""
import math

import cv2
import numpy as np
import pytest

from oracle import cvsteer_ref as ref
from tests import f64ref as R
from tests import util
from tests.util import synth

F32 = np.float32
TINY_SHAPES = [(1, 1), (1, 2), (2, 3), (3, 3), (4, 5), (5, 9), (9, 4), (1, 7), (7, 2), (13, 13)]


@pytest.mark.parametrize("shape", TINY_SHAPES)
def test_mirror_filtering_is_cv2_reflect101(shape):
    img = synth(7 + shape[0], *shape).astype(np.float64)
    for fam in (2, 4):
        F = R.family(fam)
        for kx, ky in F.pairs:
            want = cv2.sepFilter2D(img, cv2.CV_64F, kx.astype(np.float64).reshape(1, -1), ky.astype(np.float64).reshape(-1, 1))
            got = R.sep64(img, kx, ky)
            assert np.max(np.abs(got - want)) <= 6e-14 * np.abs(img).max(), (fam, shape)


def test_fast_atan2_is_cv_cart_to_polar():
    """The float64 polynomial is cv2.cartToPolar's angle to float32 evaluation error (< 1e-6 rad), and up to 1.67e-4 rad away
    from the true atan2 -- which is why the reference cannot use np.arctan2."""
    rng = np.random.default_rng(1)
    x = rng.standard_normal(2_000_000).astype(F32) * rng.choice([1e-3, 1.0, 1e3], 2_000_000).astype(F32)
    y = rng.standard_normal(2_000_000).astype(F32)
    _, cv = cv2.cartToPolar(x, y)
    mine = R.fast_atan2(y, x)
    assert np.max(R.circ_diff(cv.reshape(-1), mine, 2 * np.pi)) <= min(1e-6, R.EPS_ATAN)   # cv evaluates it in float32
    d = float(np.max(R.circ_diff(mine, np.arctan2(y.astype(np.float64), x.astype(np.float64)) % (2 * np.pi), 2 * np.pi)))
    assert 1.6e-4 <= d <= 1.7e-4, d
    # the quadrant logic at the axes and at the signed zeros
    for yy, xx, want in ((0.0, 1.0, 0.0), (1.0, 0.0, math.pi / 2), (0.0, -1.0, math.pi), (-1.0, 0.0, 1.5 * math.pi),
                         (-0.0, 1.0, 0.0), (0.0, 0.0, 0.0)):
        assert abs(float(R.fast_atan2(yy, xx)) - want) < 1e-12, (yy, xx)


def test_cv_polar_to_cart_error_figure():
    """EPS_POLAR_TO_CART is cv2.polarToCart's measured error on [-4, 4]."""
    th = np.random.default_rng(2).uniform(-4, 4, 2_000_000).astype(F32)
    c, s = cv2.polarToCart(None, th)
    t = th.astype(np.float64)
    err = max(np.abs(c.reshape(-1) - np.cos(t)).max(), np.abs(s.reshape(-1) - np.sin(t)).max())
    assert err <= R.EPS_POLAR_TO_CART, err


def test_g2_forms_are_the_projection_of_the_energy():
    """G2.cpp:93-95 are the lowest Fourier terms of g2(theta)^2 + h2(theta)^2: the same projection defines the G4 forms."""
    wg, wh = R._g2_weights()
    proj = R.projected_forms(wg, wh)
    for k in range(3):
        want = {(i, j): q for i, j, q in R.G2_FORMS[k]}
        got = {(i, j): q for i, j, q in proj[k]}
        assert set(want) == set(got), k
        for key in want:
            assert abs(want[key] - got[key]) < 1e-12, (k, key)


# --------------------------------------------------------------------------------------------------------------------------
# the cv2 float32 oracle passes every check at every pixel
# --------------------------------------------------------------------------------------------------------------------------
def _check_g2(o, img, theta_map, scalars, F=None, tag=""):
    F = F or R.family(2)
    frac = 0.01 if img.size >= 1000 else None     # frames of a few pixels have no determined orientation
    B, S = R.basis(img, F)
    beta = R.basis_bound(S, F)
    for q, n in enumerate(F.names):
        R.check(f"oracle{tag} {n}", getattr(o, n), (B[q], beta[q]))
    ori = R.orientation(B, beta, F)
    for k in ("c1", "c2", "c3", "strength"):
        R.check(f"oracle{tag} {k}", getattr(o, k), ori[k])
    R.check_angle(f"oracle{tag} theta", o.theta, ori["theta"], np.pi, max_excluded_frac=frac)
    for th in [o.theta, theta_map]:
        w = o.steer_map_full(th)
        eps = R.EPS_POLAR_TO_CART
        g, h = R.steer(B, beta, F, th, eps)
        R.check(f"oracle{tag} map g2", w[0], g)
        R.check(f"oracle{tag} map h2", w[1], h)
        R.check(f"oracle{tag} map e", w[2], R.energy(ori, th, eps))
        m, p = R.mag_phase(g, h)
        R.check(f"oracle{tag} map magnitude", w[3], m)
        R.check_angle(f"oracle{tag} map phase", w[4], p, 2 * np.pi, max_excluded_frac=frac)
        fd = R.find(m, p, eps)
        R.check(f"oracle{tag} edges", ref.find_edges(w[3], w[4]), fd["edges"])
        R.check(f"oracle{tag} dark", ref.find_dark_lines(w[3], w[4]), fd["lines_dark"])
        R.check(f"oracle{tag} bright", ref.find_bright_lines(w[3], w[4]), fd["lines_bright"])
    for t in scalars:
        w = o.steer_scalar_full(t)
        g, h = R.steer(B, beta, F, F32(t), R.EPS_SINCOS_HOST)
        R.check(f"oracle{tag} scalar g2", w[0], g)
        R.check(f"oracle{tag} scalar h2", w[1], h)
        R.check(f"oracle{tag} scalar e", w[2], R.energy(ori, F32(t), R.EPS_SINCOS_HOST))
        m, p = R.mag_phase(g, h)
        R.check(f"oracle{tag} scalar magnitude", w[3], m)
        R.check_angle(f"oracle{tag} scalar phase", w[4], p, 2 * np.pi, max_excluded_frac=frac)


def _check_g4(o4, img, theta_map, scalars, tag=""):
    F = R.family(4)
    frac = 0.01 if img.size >= 1000 else None
    B, S = R.basis(img, F)
    beta = R.basis_bound(S, F)
    for q, n in enumerate(F.names):
        R.check(f"oracle{tag} {n}", getattr(o4, n), (B[q], beta[q]))
    g4m = o4.steer_map_full(theta_map)
    g, h = R.steer(B, beta, F, theta_map, R.EPS_POLAR_TO_CART)
    R.check(f"oracle{tag} map g4", g4m[0], g)
    R.check(f"oracle{tag} map h4", g4m[1], h)
    m, p = R.mag_phase(g, h)
    R.check(f"oracle{tag} map magnitude4", g4m[2], m)
    R.check_angle(f"oracle{tag} map phase4", g4m[3], p, 2 * np.pi, max_excluded_frac=frac)
    for t in scalars:
        gs, hs = o4.steer_scalar(t)
        g, h = R.steer(B, beta, F, F32(t), R.EPS_SINCOS_HOST)
        R.check(f"oracle{tag} scalar g4", gs, g)
        R.check(f"oracle{tag} scalar h4", hs, h)


def _frames():
    fish = np.load(util.__file__.replace("util.py", "golden/fish_fixture.npz"))["fish"]
    return [("130x131", synth(11, 130, 131)), ("3x5", synth(12, 3, 5)), ("1x1", synth(13, 1, 1)),
            ("fish", np.asarray(fish, np.float32))]


@pytest.mark.parametrize("which", ["130x131", "3x5", "1x1", "fish"])
def test_oracle_passes_every_check(which):
    img = dict(_frames())[which]
    rng = np.random.default_rng(3)
    tmap = rng.uniform(-np.pi, np.pi, img.shape).astype(F32)
    scalars = (0.7, 1.5707, 1.5709, -1.5707, -1.5709)
    _check_g2(ref.SteerableFiltersG2(img), img, tmap, scalars)
    _check_g4(ref.SteerableFiltersG4(img), img, tmap, scalars)
    lvl = ref.pyr_down(img)
    R.check("oracle pyr_down", lvl, R.pyr_down(img))


def test_float32_emulation_with_other_order_passes():
    """Reversed taps, separate multiply and add, and the epilogue in another order: not bit-exact with cv2, still within every
    bound -- the checks are not bit-exactness in disguise."""
    img = synth(21, 40, 57)
    F = R.family(2)

    def corr32(x, k, axis):
        k = k.astype(F32)[::-1]                 # taps in reverse order
        n = len(k) // 2
        idx = np.arange(x.shape[axis])
        acc = np.zeros_like(x, F32)
        for jj in range(len(k)):
            off = n - jj                        # reversed position -> tap offset
            src = np.take(x, [int(ref_idx) for ref_idx in _reflect101(idx + off, x.shape[axis])], axis=axis)
            acc = (acc + (src * k[jj]).astype(F32)).astype(F32)
        return acc

    planes = [corr32(corr32(img, kx, 1), ky, 0) for kx, ky in F.pairs]
    B, S = R.basis(img, F)
    beta = R.basis_bound(S, F)
    assert not np.array_equal(planes[0], ref.SteerableFiltersG2(img).g2a)
    for q in range(F.nb):
        R.check(f"emulated {F.names[q]}", planes[q], (B[q], beta[q]))
    ori = R.orientation(B, beta, F)
    cs = []
    for terms in R.G2_FORMS:
        acc = np.zeros_like(img)
        for i, j, q in reversed(terms):
            acc = (acc + (F32(q) * (planes[i] * planes[j]).astype(F32)).astype(F32)).astype(F32)
        cs.append(acc)
    for k, c in zip(("c1", "c2", "c3"), cs):
        R.check(f"emulated {k}", c, ori[k])


def _reflect101(p, n):
    p = np.asarray(p).copy()
    if n == 1:
        return np.zeros_like(p)
    while np.any((p < 0) | (p >= n)):
        p = np.where(p < 0, -p, p)
        p = np.where(p >= n, 2 * (n - 1) - p, p)
    return p


# --------------------------------------------------------------------------------------------------------------------------
# defects are rejected
# --------------------------------------------------------------------------------------------------------------------------
def _bf16(a):
    b = np.ascontiguousarray(a, F32).view(np.uint32)
    b = ((b + 0x7FFF + ((b >> 16) & 1)) & 0xFFFF0000).astype(np.uint32)
    return b.view(F32)


def _mutants(img):
    """name -> (quantity, mutated float32 plane, want from the clean oracle, old-helper verdict kind)."""
    o = ref.SteerableFiltersG2(img)
    out = {}

    m = ref.SteerableFiltersG2.__new__(ref.SteerableFiltersG2)
    m.__dict__.update({k: v.copy() for k, v in o.__dict__.items() if k in ("g1", "g2", "g3", "h1", "h2", "h3", "h4")})
    m.g1[0, 0] *= F32(1 + 1e-3)
    m.setup(img)
    out["outer tap x (1 + 1e-3)"] = ("g2a", m.g2a)

    th = np.arctan2(o.c3.astype(np.float64), o.c2.astype(np.float64)) % (2 * np.pi)
    out["theta_d from np.arctan2"] = ("theta", (0.5 * R.wrap(th)).astype(F32))

    ct, st = cv2.polarToCart(None, o.theta)
    ct, st = _bf16(ct), _bf16(st)
    ct2, ct3, st2, st3 = ct * ct, ct * ct * ct, st * st, st * st * st
    out["sin/cos rounded to bf16"] = ("g2", (ct2 * o.g2a - F32(2) * ct * st * o.g2b + st2 * o.g2c).astype(F32))

    a, b, c = o.g2a, o.g2b, o.g2c
    ha, hb, hc, hd = o.h2a, o.h2b, o.h2c, o.h2d
    c3 = ((-(a * b)) - b * c - F32(0.9375 * (1 + 1e-3)) * (hc * hd + ha * hb) - F32(1.6875) * (hb * hc)
          - F32(0.1875) * (ha * hd)).astype(F32)
    out["c3 coefficient x (1 + 1e-3)"] = ("c3", c3)

    pad = o.width if hasattr(o, "width") else 4
    big = cv2.copyMakeBorder(img, pad, pad, 0, pad, cv2.BORDER_REFLECT_101)
    big = cv2.copyMakeBorder(big, 0, 0, pad, 0, cv2.BORDER_REFLECT)          # reflect, not reflect-101, on the left
    g2a = cv2.sepFilter2D(big, cv2.CV_32F, o.g1.reshape(1, -1), o.g2.reshape(-1, 1))[pad:-pad, pad:-pad]
    out["reflect on the left border"] = ("g2a", g2a)
    return o, out


def test_mutations_are_rejected_and_old_verdicts_recorded():
    img = synth(31, 130, 131)
    F = R.family(2)
    B, S = R.basis(img, F)
    beta = R.basis_bound(S, F)
    ori = R.orientation(B, beta, F)
    o, muts = _mutants(img)
    th = o.theta
    rng = util.basis_range([getattr(o, k) for k in o.PLANES])
    want = {n: (B[q], beta[q]) for q, n in enumerate(F.names)}
    want.update({k: ori[k] for k in ("c2", "c3", "theta")})
    want["g2"] = R.steer(B, beta, F, th, R.EPS_POLAR_TO_CART)[0]
    clean = {"g2a": o.g2a, "c3": o.c3, "theta": o.theta, "g2": o.steer_map(th)[0]}
    verdicts = {}
    for name, (qty, got) in muts.items():
        if qty == "theta":
            r, _ = R.angle_ratio(got, *want[qty], np.pi)
        else:
            r = R.err_ratio(got, *want[qty])
        n0 = len(util.RECORDS)
        try:
            if qty == "theta":
                util.assert_angle_close(got, clean[qty], o.strength, np.pi, name)
            elif qty == "c3":
                util.assert_close_range(got, clean[qty], ("own", rng), name)
            else:
                util.assert_close_range(got, clean[qty], rng, name)
            old = "accepted"
        except AssertionError:
            old = "rejected"
        finally:
            del util.RECORDS[n0:]
        verdicts[name] = (r, old)
        R.record("f64mutation", f"{name}: {qty} (old helpers: {old})", r, 0, got.size)
        assert r > 1.0, f"{name}: the float64 bound did not reject it (err/bound {r:.3g})"
    print({k: (f"{r:.3g}", v) for k, (r, v) in verdicts.items()})
    # the two defects the range / threshold helpers of tests/util.py let through
    assert verdicts["outer tap x (1 + 1e-3)"][1] == "accepted"
    assert verdicts["theta_d from np.arctan2"][1] == "accepted"
