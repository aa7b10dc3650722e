"""Shared helpers for the parity tests.

Tolerances (BASELINE.json north_star): max abs error <= 1e-4 of the basis range for filter outputs, angle error
<= 1e-3 rad where strength exceeds a threshold.  Angles are compared on the circle (period pi for the dominant
orientation, 2 pi for phase)."""
import hashlib

import numpy as np

BASIS_RTOL = 1e-4      # of the basis range
ANGLE_TOL = 1e-3       # rad

# Every comparison made through the helpers below is recorded here; tests/conftest.py writes the per-quantity maxima to
# gpurun_out/parity_achieved.json at the end of a GPU session (copied to profiles/parity.json by hand).
RECORDS = []


def _record(kind, name, err, tol, scale, n):
    RECORDS.append({"kind": kind, "name": name, "err": float(err), "tol": float(tol), "scale": float(scale), "n": int(n)})


def synth(seed, rows, cols):
    """SURVEY section 8d synthetic input: fp32 uniform[0,255) from default_rng(seed)."""
    return np.random.default_rng(seed).uniform(0, 255, (rows, cols)).astype(np.float32)


def fish_oracle_planes(fish):
    """The oracle's float-level outputs on the fish image, keyed as in tests/golden/fish_oracle_cv2_4_13.json: G2/H2 basis,
    c1..c3, theta, strength, steer at theta (g2, h2, e, magnitude, phase), G4/H4 basis, G4 steer at 0.3 and at theta,
    and pyramid levels 1..4."""
    from oracle import cvsteer_ref as ref
    f2, (g2, h2, e, mag, phase) = ref.g2_full(fish)
    out = {k: getattr(f2, k) for k in ref.SteerableFiltersG2.PLANES}
    out.update(c1=f2.c1, c2=f2.c2, c3=f2.c3, theta=f2.theta, strength=f2.strength,
               g2=g2, h2=h2, e=e, magnitude=mag, phase=phase)
    f4 = ref.SteerableFiltersG4(fish)
    out.update({k: getattr(f4, k) for k in ref.SteerableFiltersG4.PLANES})
    g4s, h4s = f4.steer_scalar(0.3)
    g4m, h4m, mag4, ph4 = f4.steer_map_full(f2.theta)
    out.update(g4_s03=g4s, h4_s03=h4s, g4_map=g4m, h4_map=h4m, mag4=mag4, phase4=ph4)
    for i, l in enumerate(ref.pyramid(fish, 5)[1:], 1):
        out[f"pyr{i}"] = l
    return out


def plane_digest(a):
    """SHA-256 of the array's bytes in C order."""
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def assert_matches_golden(name, got, entry):
    """`got` is bit for bit the committed plane `entry` of tests/golden/fish_oracle_cv2_4_13.json: float32, same shape,
    the same values at the stored sample positions, and the same SHA-256 over every pixel."""
    assert got.dtype == np.float32 and list(got.shape) == entry["shape"], (name, got.dtype, got.shape, entry["shape"])
    vals = np.ascontiguousarray(got).reshape(-1)[np.asarray(entry["sample_index"])]
    want = np.asarray(entry["sample"], np.float32)
    assert np.array_equal(vals, want), \
        f"{name}: sampled values differ from the committed ones by up to {float(np.max(np.abs(vals - want))):.3e}"
    assert plane_digest(got) == entry["sha256"], f"{name}: differs from the committed plane (the sampled values agree)"


def basis_range(planes):
    return float(max(p.max() for p in planes) - min(p.min() for p in planes))


def own_range(want, basis_rng):
    """Range of a QUADRATIC quantity (c1..c3, strength, energy) for its own tolerance: max - min of the oracle's plane.
    Degenerate planes (constant images: strength == 0 everywhere) fall back to rtol x basis_range^2 so that rounding
    residue of the filters (taps do not sum to exactly zero) is not compared at zero tolerance."""
    w = np.asarray(want, dtype=np.float64)
    ptp = float(w.max() - w.min()) if w.size else 0.0
    return max(ptp, BASIS_RTOL * basis_rng * basis_rng)


def assert_close_range(got, want, rng, name="", rtol=BASIS_RTOL):
    """max abs error <= rtol x rng.  rng = ("own", basis_range): the quantity's OWN range (see own_range)."""
    assert got.shape == want.shape, (name, got.shape, want.shape)
    if isinstance(rng, tuple):
        rng = own_range(want, rng[1])
    err = float(np.max(np.abs(got.astype(np.float64) - want.astype(np.float64)))) if got.size else 0.0
    _record("range", name, err, rtol * rng, rng, got.size)
    assert err <= rtol * rng, f"{name}: max abs err {err:.3e} > {rtol:g} x range {rng:.3e}"
    return err


def circ_diff(a, b, period):
    d = np.abs(a.astype(np.float64) - b.astype(np.float64)) % period
    return np.minimum(d, period - d)


def assert_angle_close(got, want, weight, period, name="", tol=ANGLE_TOL, thresh_frac=1e-3):
    """Compare angles where `weight` (strength / magnitude) exceeds thresh_frac of its max."""
    m = weight > thresh_frac * float(weight.max()) if weight.size and weight.max() > 0 else np.zeros_like(weight, bool)
    if not m.any():
        return 0.0
    err = float(circ_diff(got[m], want[m], period).max())
    _record("angle", name, err, tol, period, int(m.sum()))
    assert err <= tol, f"{name}: max angle err {err:.3e} rad > {tol:g} over {int(m.sum())} px"
    return err
