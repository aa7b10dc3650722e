"""Float64 reference of every fused quantity, with a per-pixel error bound for float32 implementations of it.

Test infrastructure, next to tests/util.py; it does not use cv2.  "Exact" means exact for the reference's own float32 taps
(oracle.cvsteer_ref.create, pinned by tests/golden/taps_default.npz) promoted to float64.

Filtering is scipy.ndimage.correlate1d(mode="mirror") in float64, rows then columns: "mirror" is BORDER_REFLECT_101, and on
these taps it equals cv2.sepFilter2D(CV_64F) to 6e-14 on every frame size, the ones smaller than the filter included.
Angles are cv::cartToPolar's (hal::fastAtan32f): a 7th-order polynomial that is up to 1.67e-4 rad away from the true atan2.
The reference evaluates that polynomial, with cv's quadrant logic, in float64 (fast_atan2); np.arctan2 would fail every
correct kernel by 100x any rounding-level bound.

Bounds.  Every check compares |got - want| with a per-pixel bound built from the error model below.  u = 2^-24 is the unit
roundoff of float32, gamma(n) = n u / (1 - n u) the bound of n successive roundings (Higham, Accuracy and Stability of
Numerical Algorithms, 2nd ed., Lemma 3.1).

- Basis planes: beta = (gamma(2 (2R+1) + 1) + fold) * S, S = (|x| (*) |t_x|) (*) |t_y| in float64.  A (2R+1)-tap pass in
  any summation order rounds each term at most 2R+1 times (the product and the adds on its path), two passes, plus one
  rounding of a steering factor folded into the column taps (G4 steer-only kernels, DESIGN section 4).  `fold` is the
  relative error of the pre-scaled shared-row taps (G2b = h3 row x g3*(g3/h3) column, G4d = h4 row x g3*(g4/h4) column,
  fill_tap_table / scale_taps_by_ratio), computed exactly from the taps; it is 0 for every other plane.
  Impulse frames (a few isolated values of 128): at most two nonzero products per pass (an impulse and its reflection), so
  each pass rounds a term at most twice, plus the folded factor: KAPPA_IMPULSE = 5.
- Quadratic forms c = sum Q_ij b_i b_j: sum |Q_ij| (|b_i| beta_j + beta_i |b_j| + beta_i beta_j) for the basis error, plus
  (nterms + 3) u sum |Q_ij| |b_i b_j| for the form's own rounding (product, accumulation depth <= nterms, the coefficient's
  float rounding, one spare for an inner add).
- hypot: the two input errors, plus 3u of the result (fma + sqrt.approx, see SQRT_APPROX_REL).
- Angles: 1.01 |d(y, x)| / |(y, x)| (arcsin(t) <= 1.01 t for t <= 0.2, and pixels whose bound exceeds EXCLUDE_RAD are not
  compared), plus the polynomial's own float32 evaluation error EPS_ATAN, plus the polynomial's jump of 1.67e-4 rad across
  |y| = |x| (ATAN_DIAGONAL_JUMP) where the inputs' error interval straddles that diagonal.  theta_d takes half of all three.
- Steering sum_i w_i(c, s) b_i: sum |w_i| beta_i + eps * sum |dw_i/dc| + |dw_i/ds|) (|b_i| + beta_i) + kappa u sum |w_i| (|b_i| +
  beta_i), eps = the sin/cos error of the form plus any angle error, kappa = weight degree + terms + 1.
- find*: d|mag| + mag * min(1, dphase + 2 eps_cos + 4 u pi) + 3u mag (cos^2 is 1-Lipschitz).
"""
from __future__ import annotations

import math
import os

import numpy as np
from scipy.ndimage import correlate1d

U = 2.0 ** -24
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def gamma(n):
    return n * U / (1.0 - n * U)


KAPPA_IMPULSE = 5
# Pixels whose angle bound exceeds this are counted, not compared: the angle of (c2, c3) or (g, h) is not determined there.
EXCLUDE_RAD = 0.1

# --- SFU and library error figures (absolute, on values in [-1, 1] unless stated) ---------------------------------------
# __sincosf / __sinf / __cosf: "For x in [-pi, pi], the maximum absolute error is 2^-21.41, and larger otherwise."
# (CUDA C++ Programming Guide 12.9, Intrinsic Functions table.)
EPS_SINCOS_FAST = 2.0 ** -21.41
# Beyond [-pi, pi]: MUFU.SIN / MUFU.COS take theta in revolutions, FMUL.RZ(theta, float(1 / 2pi)) (the SASS of every
# __sincosf here).  Round-toward-zero is off by < 1 ulp (2u relative) and float(1 / 2pi) by 0.68u relative, so the argument
# is off by up to (2u + 0.68u) |theta| rad on top of the figure above.  (families.cuh said 6e-8 |theta|, one rounding; angle
# maps in [-8, 8] on a B200 exceed that by 13 % in the steered planes.)
EPS_SINCOS_FAST_BEYOND = EPS_SINCOS_FAST
EPS_SINCOS_FAST_PER_RAD = 2 * U + abs(float(np.float32(1 / (2 * math.pi))) * 2 * math.pi - 1)
# dev::sincos_steer: minimax polynomials, 1.4e-7 for |x| <= pi/2 (device_math.cuh); libdevice sinf/cosf beyond, 2 ulp
# (CUDA C++ Programming Guide 12.9, single-precision function table) = 1.2e-7 on [-1, 1].
EPS_SINCOS_STEER = 1.4e-7
# Host std::cos(float) / std::sin(float) (glibc, <= 1 ulp) for scalar angles: 1 ulp of a value <= 1 is <= 2^-23.
EPS_SINCOS_HOST = 2.0 ** -23
# cv2.polarToCart: measured 7.06e-8 on 2 M angles in [-4, 4] (tests/test_f64ref_cpu.py re-measures it).
EPS_POLAR_TO_CART = 7.1e-8
# rcp.approx.ftz.f32: "The maximum ulp error is 1 across the full range" (PTX ISA 8.8, CUDA 12.9).
RCP_APPROX_ULP = 1
# sqrt.approx.ftz.f32: maximum relative error 2^-23 (PTX ISA 8.8, CUDA 12.9).
SQRT_APPROX_REL = 2.0 ** -23
# cv atan polynomial in float32, in radians: the ratio min/max (rcp: 2u, product: u), the polynomial at |a| <= pi/4 (four
# FMA/multiply roundings: 4u), then at most five roundings of values up to 2 pi with rounded constants (quadrant selects,
# degree -> radian, wrap: 1.5u * 2pi each, 47u): 56u, taken as 64u.  theta_d = half of it.
EPS_ATAN = 64 * U


# ==========================================================================================================================
# taps and families
# ==========================================================================================================================
def _oracle_taps(fam, width, spacing):
    from oracle import cvsteer_ref as ref
    names = ("G21", "G22", "G23", "H21", "H22", "H23", "H24") if fam == 2 else \
        ("G41", "G42", "G43", "G44", "G45", "H41", "H42", "H43", "H44", "H45", "H46")
    return [ref.create(width, spacing, getattr(ref, n)).reshape(-1) for n in names]


def default_taps(fam):
    """The reference-default taps as committed in tests/golden/taps_default.npz (API order)."""
    z = np.load(os.path.join(GOLDEN, "taps_default.npz"))
    keys = ("g1", "g2", "g3", "h1", "h2", "h3", "h4") if fam == 2 else \
        tuple("G4_" + k for k in ("g1", "g2", "g3", "g4", "g5", "h1", "h2", "h3", "h4", "h5", "h6"))
    return [z[k].astype(np.float32) for k in keys]


def _scaled(src, num, den):
    """scale_taps_by_ratio (cvsteer_b200/csrc/taps.cpp): src * (num[k] / den[k]) at den's largest |tap|, rounded to float."""
    k = int(np.argmax(np.abs(den)))
    r = float(num[k]) / float(den[k]) if den[k] != 0 else 0.0
    return (src.astype(np.float64) * r).astype(np.float32)


def _fold_rel(row_ref, col_ref, row_k, col_k):
    """max over taps of |row_k[i] col_k[j] / (row_ref[i] col_ref[j]) - 1|: the relative error of a product of pre-scaled taps."""
    want = np.outer(row_ref.astype(np.float64), col_ref.astype(np.float64))
    got = np.outer(row_k.astype(np.float64), col_k.astype(np.float64))
    nz = want != 0
    assert np.all(got[~nz] == 0)
    return float(np.max(np.abs(got[nz] / want[nz] - 1.0)))


def _g2_weights():
    # (coef, p, q): w = coef c^p s^q.  G2.cpp:140-144
    g = [(1, 2, 0), (-2, 1, 1), (1, 0, 2)]
    h = [(1, 3, 0), (-3, 2, 1), (3, 1, 2), (-1, 0, 3)]
    return g, h


def _g4_weights():
    # G4.cpp:116-121
    g = [(1, 4, 0), (-4, 3, 1), (6, 2, 2), (-4, 1, 3), (1, 0, 4)]
    h = [(1, 5, 0), (-5, 4, 1), (10, 3, 2), (-10, 2, 3), (5, 1, 4), (-1, 0, 5)]
    return g, h


# G2.cpp:93-95 as (i, j, coefficient) over the basis (g2a g2b g2c h2a h2b h2c h2d) = 0..6
G2_FORMS = (
    ((1, 1, .5), (0, 2, .25), (0, 0, .375), (2, 2, .375), (3, 3, .3125), (6, 6, .3125), (4, 4, .5625), (5, 5, .5625),
     (3, 5, .375), (4, 6, .375)),
    ((0, 0, .5), (2, 2, -.5), (3, 3, .46875), (6, 6, -.46875), (4, 4, .28125), (5, 5, -.28125), (3, 5, .1875),
     (4, 6, -.1875)),
    ((0, 1, -1.), (1, 2, -1.), (5, 6, -.9375), (3, 4, -.9375), (4, 5, -1.6875), (3, 6, -.1875)),
)


def projected_forms(wg, wh, n=32):
    """C1, C2, C3 of E(theta) = (sum w_i b_i)^2 + (sum v_j h_j)^2 as quadratic forms over the basis: E projected on 1,
    cos 2theta, sin 2theta at n angles, in float64 (exact for these trigonometric polynomials of degree <= 10 when n = 32)."""
    nb = len(wg) + len(wh)
    Q = np.zeros((3, nb, nb))
    for t in range(n):
        th = 2 * np.pi * t / n
        c, s = math.cos(th), math.sin(th)
        w = np.array([k * c ** p * s ** q for k, p, q in wg] + [0.0] * len(wh))
        v = np.array([0.0] * len(wg) + [k * c ** p * s ** q for k, p, q in wh])
        E = np.outer(w, w) + np.outer(v, v)
        Q[0] += E / n
        Q[1] += 2 * E * math.cos(2 * th) / n
        Q[2] += 2 * E * math.sin(2 * th) / n
    forms = []
    for k in range(3):
        terms = []
        for i in range(nb):
            for j in range(i, nb):
                coef = Q[k, i, i] if i == j else Q[k, i, j] + Q[k, j, i]
                if abs(coef) > 1e-12:
                    terms.append((i, j, float(coef)))
        forms.append(tuple(terms))
    return tuple(forms)


class Family:
    """Taps, basis pairs, steering weights and orientation forms of one filter family at (width, spacing)."""

    def __init__(self, fam, width=None, spacing=None, taps=None):
        self.fam = fam
        self.width = width if width is not None else (4 if fam == 2 else 6)
        self.spacing = spacing if spacing is not None else (0.67 if fam == 2 else 0.5)
        self.R = self.width
        if taps is None:
            default = (self.width, self.spacing) == ((4, 0.67) if fam == 2 else (6, 0.5))
            taps = default_taps(fam) if default else _oracle_taps(fam, self.width, self.spacing)
        self.taps = [np.asarray(t, np.float32) for t in taps]
        t = self.taps
        if fam == 2:
            g1, g2, g3, h1, h2, h3, h4 = t
            # (row taps = kernelX, column taps = kernelY): G2.cpp:62-68
            self.pairs = [(g1, g2), (g3, g3), (g2, g1), (h1, h2), (h4, h3), (h3, h4), (h2, h1)]
            self.names = ("g2a", "g2b", "g2c", "h2a", "h2b", "h2c", "h2d")
            self.wg, self.wh = _g2_weights()
            self.forms = G2_FORMS
            self.fold = [0.0] * 7
            self.fold[1] = _fold_rel(g3, g3, h3, _scaled(g3, g3, h3))          # G2b from the h3 row plane
        else:
            g1, g2, g3, g4, g5, h1, h2, h3, h4, h5, h6 = t
            # G4.cpp:69-80
            self.pairs = [(g1, g2), (g3, g4), (g5, g5), (g4, g3), (g2, g1),
                          (h1, h2), (h3, h4), (h5, h6), (h6, h5), (h4, h3), (h2, h1)]
            self.names = ("g4a", "g4b", "g4c", "g4d", "g4e", "h4a", "h4b", "h4c", "h4d", "h4e", "h4f")
            self.wg, self.wh = _g4_weights()
            self.forms = projected_forms(self.wg, self.wh)
            self.fold = [0.0] * 11
            self.fold[3] = _fold_rel(g4, g3, h4, _scaled(g3, g4, h4))          # G4d from the h4 row plane
        self.ng = len(self.wg)
        self.nb = len(self.pairs)


_FAMILIES = {}


def family(fam, width=None, spacing=None):
    key = (fam, width, spacing)
    if key not in _FAMILIES:
        _FAMILIES[key] = Family(fam, width, spacing)
    return _FAMILIES[key]


# ==========================================================================================================================
# filtering
# ==========================================================================================================================
def sep64(img, kx, ky):
    """cv::sepFilter2D(img, CV_64F, kx, ky) with BORDER_REFLECT_101, in float64: rows (kx along x), then columns."""
    x = np.asarray(img, np.float64)
    r = correlate1d(x, np.asarray(kx, np.float64), axis=1, mode="mirror")
    return correlate1d(r, np.asarray(ky, np.float64), axis=0, mode="mirror")


def basis(img, F):
    """(B, S): the exact basis planes [nb, H, W] and S = (|x| (*) |t_x|) (*) |t_y| per plane, both float64."""
    a = np.abs(np.asarray(img, np.float64))
    B = np.stack([sep64(img, kx, ky) for kx, ky in F.pairs])
    S = np.stack([sep64(a, np.abs(kx), np.abs(ky)) for kx, ky in F.pairs])
    return B, S


def basis_bound(S, F, impulse=False):
    """Per-pixel bound of a float32 basis plane (module docstring)."""
    k = gamma(KAPPA_IMPULSE) if impulse else gamma(2 * (2 * F.R + 1) + 1)
    return np.stack([(k + F.fold[q]) * S[q] for q in range(F.nb)])


# ==========================================================================================================================
# angles
# ==========================================================================================================================
_P1, _P3, _P5, _P7 = 0.9997878412794807, -0.3258083974640975, 0.1555786518463281, -0.04432655554792128


def fast_atan2(y, x):
    """cv::fastAtan2 / cartToPolar's angle (hal::fastAtan32f) in float64, in radians on [0, 2 pi): the polynomial in
    min/max and cv's quadrant logic (ay > ax: 90 - a; x < 0: 180 - a; y < 0: 360 - a)."""
    y = np.asarray(y, np.float64)
    x = np.asarray(x, np.float64)
    ax, ay = np.abs(x), np.abs(y)
    mx, mn = np.maximum(ax, ay), np.minimum(ax, ay)
    c = mn / (mx + 2.220446049250313e-16)
    c2 = c * c
    a = (((_P7 * c2 + _P5) * c2 + _P3) * c2 + _P1) * c
    a = np.where(ay > ax, np.pi / 2 - a, a)
    a = np.where(x < 0, np.pi - a, a)
    a = np.where(y < 0, 2 * np.pi - a, a)
    return a


def wrap(a):
    """SteerableFilters::wrap: (pi, 2 pi) -> (-pi, 0)."""
    return np.where(a > np.pi, a - 2 * np.pi, a)


def circ_diff(a, b, period):
    d = np.abs(np.asarray(a, np.float64) - np.asarray(b, np.float64)) % period
    return np.minimum(d, period - d)


# The polynomial is not continuous across |y| = |x|: at c = 1 it gives P1 + P3 + P5 + P7 = pi/4 - 8.3e-5, and the branch
# `90 - a` gives pi/4 + 8.3e-5.  Inputs whose error interval straddles the diagonal may land on either side.
ATAN_DIAGONAL_JUMP = 2 * (math.pi / 4 - (_P1 + _P3 + _P5 + _P7))


def angle_bound(dy, dx, y, x, scale=1.0):
    """Bound of the angle of (y, x) computed from inputs within (dy, dx), times `scale` (0.5 for theta_d): the condition
    number, the float32 evaluation, and the polynomial's jump at the diagonal where the inputs may straddle it."""
    r = np.hypot(y, x)
    with np.errstate(divide="ignore", invalid="ignore"):
        cond = np.where(r > 0, 1.01 * (dy + dx) / r, np.inf)
    jump = np.where(np.abs(np.abs(y) - np.abs(x)) <= (dy + dx) * (1 + 1e-6) + 4 * U * r, ATAN_DIAGONAL_JUMP, 0.0)
    return scale * (cond + EPS_ATAN + jump)


# ==========================================================================================================================
# epilogue
# ==========================================================================================================================
def _form(terms, B, beta):
    v = np.zeros(B.shape[1:])
    d = np.zeros(B.shape[1:])
    mag = np.zeros(B.shape[1:])
    aB = np.abs(B)
    for i, j, q in terms:
        v += q * B[i] * B[j]
        d += abs(q) * (aB[i] * beta[j] + beta[i] * aB[j] + beta[i] * beta[j])
        mag += abs(q) * (aB[i] + beta[i]) * (aB[j] + beta[j])
    return v, d + (len(terms) + 3) * U * mag


def orientation(B, beta, F):
    """c1, c2, c3, strength, theta_d (each a (value, bound) pair; theta's bound is in rad and +inf where undetermined)."""
    (c1, d1), (c2, d2), (c3, d3) = (_form(t, B, beta) for t in F.forms)
    st = np.hypot(c2, c3)
    dst = d2 + d3 + 3 * U * (st + d2 + d3)
    th = 0.5 * wrap(fast_atan2(c3, c2))
    dth = angle_bound(d3, d2, c3, c2, 0.5)
    return dict(c1=(c1, d1), c2=(c2, d2), c3=(c3, d3), strength=(st, dst), theta=(th, dth))


def _weights(spec, c, s, eps):
    """Values and |dw/dc| + |dw/ds| (at |c| + eps, |s| + eps: a bound over the whole error interval) of the weights."""
    w, dw = [], []
    ac, as_ = np.abs(c) + eps, np.abs(s) + eps
    for k, p, q in spec:
        w.append(k * c ** p * s ** q)
        d = 0.0
        if p:
            d = d + abs(k) * p * ac ** (p - 1) * as_ ** q
        if q:
            d = d + abs(k) * q * ac ** p * as_ ** (q - 1)
        dw.append(d)
    return w, dw


def _steer_sum(spec, planes, betas, c, s, eps):
    w, dw = _weights(spec, c, s, eps)
    deg = max(p + q for _, p, q in spec)
    kappa = deg + len(spec) + 1
    v = sum(wi * b for wi, b in zip(w, planes))
    d = 0.0
    for wi, dwi, b, be in zip(w, dw, planes, betas):
        a = np.abs(b) + be
        d = d + np.abs(wi) * be + eps * dwi * a + kappa * U * np.abs(wi) * a
    return v, d


def steer(B, beta, F, theta, eps_sc, dtheta=0.0):
    """G(theta), H(theta) from the exact basis at the angle the kernel used (float64 cos / sin of it).  eps_sc: the form's
    sin/cos error (scalar or per pixel); dtheta: any error of the angle itself (the reference's theta_d for kernels that
    steer to their own theta_d without storing it)."""
    th = np.asarray(theta, np.float64)
    c, s = np.cos(th), np.sin(th)
    eps = eps_sc + dtheta
    ng = F.ng
    g = _steer_sum(F.wg, B[:ng], beta[:ng], c, s, eps)
    h = _steer_sum(F.wh, B[ng:], beta[ng:], c, s, eps)
    return g, h


def energy(o, theta, eps_sc, dtheta=0.0):
    """c1 + c2 cos 2theta + c3 sin 2theta (G2.cpp:174-176) at a given angle; the kernel forms cos 2t / sin 2t from its own
    c, s (c^2 - s^2, 2cs: 3 eps + 2u) or directly (eps)."""
    th = np.asarray(theta, np.float64)
    C2, S2 = np.cos(2 * th), np.sin(2 * th)
    (c1, d1), (c2, d2), (c3, d3) = o["c1"], o["c2"], o["c3"]
    e = c1 + c2 * C2 + c3 * S2
    e2 = 3 * eps_sc + 2 * U + 2 * dtheta
    a1, a2, a3 = np.abs(c1) + d1, np.abs(c2) + d2, np.abs(c3) + d3
    d = d1 + np.abs(C2) * d2 + np.abs(S2) * d3 + (a2 + a3) * e2 + 4 * U * (a1 + a2 + a3)
    return e, d


def energy_dominant(o):
    """E(theta_d) = c1 + strength (the fused kernels' form of G2.cpp:174-176 at theta_d)."""
    (c1, d1), (st, dst) = o["c1"], o["strength"]
    return c1 + st, d1 + dst + 2 * U * (np.abs(c1) + st + d1 + dst)


def mag_phase(g, h):
    """magnitude, phase = wrap(fastAtan(h, g)) (G2.cpp:107-112)."""
    (gv, dg), (hv, dh) = g, h
    m = np.hypot(gv, hv)
    dm = dg + dh + 3 * U * (m + dg + dh)
    ph = wrap(fast_atan2(hv, gv))
    dph = angle_bound(dh, dg, hv, gv)
    return (m, dm), (ph, dph)


def phase_weight(phase, phi, signum):
    """G2.cpp:179-186 in float64."""
    err = np.abs(phase - phi) if signum else np.abs(np.abs(phase) - abs(phi))
    err = np.minimum(err, 2 * np.pi - err)
    lam = np.cos(err) ** 2
    return np.where(np.abs(err) > np.pi / 2, 0.0, lam)


FIND = {"edges": (math.pi / 2, False), "lines_dark": (0.0, True), "lines_bright": (math.pi, True)}


def find(mag, phase, eps_cos=EPS_SINCOS_FAST):
    """edges / dark / bright lines of (magnitude, phase) (G2.cpp:201-212) with bounds."""
    (m, dm), (ph, dph) = mag, phase
    out = {}
    for k, (phi, sg) in FIND.items():
        v = m * phase_weight(ph, phi, sg)
        d = dm + (m + dm) * np.minimum(1.0, dph + 2 * eps_cos + 4 * U * np.pi) + 3 * U * (m + dm)
        out[k] = (v, d)
    return out


def g4_orientation(B, beta, F):
    """G4 theta_d / strength: the projection of E(theta) = G4(theta)^2 + H4(theta)^2 on cos 2theta / sin 2theta."""
    return orientation(B, beta, F)


def sincos_eps_fast(theta):
    """|error| of __sincosf at theta (per pixel)."""
    a = np.abs(np.asarray(theta, np.float64))
    return np.where(a <= np.pi, EPS_SINCOS_FAST, EPS_SINCOS_FAST_BEYOND + EPS_SINCOS_FAST_PER_RAD * a)


# ==========================================================================================================================
# pyramid
# ==========================================================================================================================
_PYR = np.array([1, 4, 6, 4, 1], np.float64) / 16


def pyr_down(img):
    """cv::pyrDown in float64: [1 4 6 4 1]/16 both ways, BORDER_REFLECT_101, even samples; bound gamma(10) S (two 5-term
    passes, power-of-two scale)."""
    x = np.asarray(img, np.float64)
    v = sep64(x, _PYR, _PYR)[::2, ::2]
    S = sep64(np.abs(x), _PYR, _PYR)[::2, ::2]
    return v, gamma(10) * S


# ==========================================================================================================================
# checks
# ==========================================================================================================================
def err_ratio(got, want, bound):
    """max |got - want| / bound over the pixels (0/0 counts as 0; anything over a zero bound as inf)."""
    e = np.abs(np.asarray(got, np.float64) - want)
    with np.errstate(divide="ignore", invalid="ignore"):
        r = np.where(e == 0, 0.0, e / bound)
    r = np.where(np.isnan(np.asarray(got, np.float64)), np.inf, r)
    return float(r.max()) if r.size else 0.0


def angle_ratio(got, want, bound, period):
    """(max circular err / bound over the determined pixels, number of pixels excluded for conditioning)."""
    keep = bound <= EXCLUDE_RAD
    e = circ_diff(got, want, period)
    with np.errstate(divide="ignore", invalid="ignore"):
        r = np.where(e == 0, 0.0, e / bound)
    r = np.where(keep, r, 0.0)
    return (float(r.max()) if r.size else 0.0), int((~keep).sum())


def record(kind, name, ratio, excluded, n):
    from tests.util import RECORDS
    RECORDS.append({"kind": kind, "name": name, "err": float(ratio), "tol": 1.0, "scale": 1.0, "n": int(n),
                    "excluded": int(excluded)})


def check(name, got, want_bound, kind="f64bound"):
    want, bound = want_bound
    got = np.asarray(got)
    assert got.shape == np.shape(want), (name, got.shape, np.shape(want))
    r = err_ratio(got, want, bound)
    record(kind, name, r, 0, got.size)
    assert r <= 1.0, f"{name}: max err/bound {r:.3g}"
    return r


def check_angle(name, got, want_bound, period, max_excluded_frac=None, kind="f64bound"):
    want, bound = want_bound
    got = np.asarray(got)
    assert got.shape == np.shape(want), (name, got.shape, np.shape(want))
    r, nx = angle_ratio(got, want, bound, period)
    record(kind, name, r, nx, got.size)
    assert r <= 1.0, f"{name}: max angle err/bound {r:.3g} ({nx} px excluded)"
    if max_excluded_frac is not None:
        assert nx <= max_excluded_frac * got.size, f"{name}: {nx} of {got.size} px excluded for conditioning"
    return r, nx
