"""Parity of the class surface (host arrays through the C ABI) against the oracle -- GPU."""
import cv2
import numpy as np
import pytest

import cvsteer_b200 as cb
from cvsteer_b200 import capi
from oracle import cvsteer_ref as ref
from tests.util import (ANGLE_TOL, assert_angle_close, assert_close_range, basis_range, synth)

pytestmark = pytest.mark.gpu

STATE = ("g2a", "g2b", "g2c", "h2a", "h2b", "h2c", "h2d")


def _check_state(f, o, name=""):
    rng = basis_range([getattr(o, k) for k in STATE])
    for k in STATE:
        assert_close_range(getattr(f, k), getattr(o, k), rng, f"{name}{k}")
    # c1..c3 and strength are quadratic in the basis: tolerance relative to range^2
    for k in ("c1", "c2", "c3"):
        assert_close_range(getattr(f, k), getattr(o, k), ("own", rng), f"{name}{k}")
    assert_close_range(f.getDominantOrientationStrength(), o.strength, ("own", rng), f"{name}strength")
    assert_angle_close(f.getDominantOrientationAngle(), o.theta, o.strength, np.pi, f"{name}theta")
    th = f.getDominantOrientationAngle()
    assert th.min() >= -np.pi / 2 - 1e-6 and th.max() <= np.pi / 2 + 1e-6
    return rng


def _check_steer(got, o, theta, rng, name=""):
    """Steering outputs vs the oracle steered with the SAME angles (so that branch-cut flips of theta_d near
    +-pi/2, which negate H2 and the phase, do not enter -- see SURVEY section 7 hard part 2)."""
    g2, h2, e, mag, ph = got
    if isinstance(theta, np.ndarray):
        w = o.steer_map_full(theta)
    else:
        w = o.steer_scalar_full(theta)
    assert_close_range(g2, w[0], rng, name + "g2")
    assert_close_range(h2, w[1], rng, name + "h2")
    assert_close_range(e, w[2], ("own", rng), name + "e")
    assert_close_range(mag, w[3], rng, name + "magnitude")
    assert_angle_close(ph, w[4], w[3], 2 * np.pi, name + "phase")
    assert ph.min() >= -np.pi - 1e-6 and ph.max() <= np.pi + 1e-6 and not np.isnan(ph).any()


def test_fish_matches_golden_vectors(fish_fixture, fish_oracle):
    """Committed cv2-4.13.0 vectors (rebuilt by the oracle and checked bit for bit against their digests)."""
    fish = fish_fixture["fish"]
    f = cb.SteerableFiltersG2(fish, 4, 0.67)  # uint8 in, like the reference callers
    rng = basis_range([fish_oracle[k] for k in STATE])
    for k in STATE:
        assert_close_range(getattr(f, k), fish_oracle[k], rng, k)
    for k in ("c1", "c2", "c3", "strength"):
        assert_close_range(getattr(f, k), fish_oracle[k], ("own", rng), k)
    assert_angle_close(f.theta, fish_oracle["theta"], fish_oracle["strength"], np.pi, "theta")
    # known-answer values of SURVEY App. C
    assert abs(float(f.g2a[92, 128]) - (-92.52432)) < 1e-3
    assert abs(float(f.h2d[92, 128]) - 42.62686) < 1e-3
    assert abs(float(f.theta[92, 128]) - 0.354760) < 1e-4
    assert abs(float(f.strength[92, 128]) - 4604.653320) < 0.05


def test_reference_gtest_on_gpu(fish_fixture):
    """TEST(cvsteer, basic) (reference test/test.cpp:70-103) with the B200 class in place of fa::SteerableFiltersG2."""
    fish = fish_fixture["fish"]
    f = cb.SteerableFiltersG2(fish, 4, 0.67)
    g2, h2, e, magnitude, phase = f.steer(f.getDominantOrientationAngle())
    maps = {"edges_gt": f.findEdges(magnitude, phase), "lines_dark_gt": f.findDarkLines(magnitude, phase),
            "lines_bright_gt": f.findBrightLines(magnitude, phase)}
    for name, m in maps.items():
        out8 = cv2.normalize(m, None, 0, 255, cv2.NORM_MINMAX, cv2.CV_8UC1)
        ok, buf = cv2.imencode(".jpg", out8)
        rec = cv2.imdecode(buf, cv2.IMREAD_GRAYSCALE)
        err = cv2.norm(rec, fish_fixture[name], cv2.NORM_L1) / float(fish.size)
        assert err <= 1.0, (name, err)


@pytest.mark.parametrize("shape", [(185, 256), (131, 257), (64, 128), (65, 129), (200, 300), (9, 9), (5, 5)])
def test_state_and_steer_vs_oracle(shape):
    img = synth(2000 + shape[0], *shape)
    o = ref.SteerableFiltersG2(img)
    f = cb.SteerableFiltersG2(img)
    rng = _check_state(f, o)
    th = f.getDominantOrientationAngle()
    _check_steer(f.steer(th), o, th, rng, "map:")
    _check_steer(f.steer(None), o, th, rng, "dominant:")
    _check_steer(f.steer(0.3), o, 0.3, rng, "scalar:")
    _check_steer(f.steer(-2.5), o, -2.5, rng, "scalar2:")
    g2, h2 = f.steer(0.3, full=False)
    assert_close_range(g2, o.steer_scalar(0.3)[0], rng, "g2-only")


@pytest.mark.parametrize("shape", [(5, 3), (3, 5), (1, 7), (7, 1), (1, 1), (2, 2), (4, 4), (3, 200), (200, 3)])
def test_tiny_images_iterated_reflect(shape):
    """Images smaller than the filter radius: OpenCV folds indices repeatedly (SURVEY App. B)."""
    img = synth(77 + shape[0] * 10 + shape[1], *shape)
    o = ref.SteerableFiltersG2(img)
    f = cb.SteerableFiltersG2(img)
    rng = max(basis_range([getattr(o, k) for k in STATE]), 1.0)
    for k in STATE:
        assert_close_range(getattr(f, k), getattr(o, k), rng, k)


def test_constant_image_and_nan_patch():
    img = np.full((40, 50), 7.0, np.float32)
    f = cb.SteerableFiltersG2(img)
    o = ref.SteerableFiltersG2(img)
    g2, h2, e, mag, ph = f.steer(None)
    assert not np.isnan(ph).any() and not np.isnan(f.theta).any()
    assert_close_range(f.g2a, o.g2a, 255.0, "g2a-const")
    img2 = synth(5, 32, 32)
    img2[10, 10] = np.nan
    f2 = cb.SteerableFiltersG2(img2)
    _, _, _, _, ph2 = f2.steer(None)
    assert not np.isnan(ph2).any()          # cv::patchNaNs(phase), G2.cpp:111
    assert ph2[10, 10] == 0.0


def test_grating_orientation_analytic():
    """Oriented sinusoid: the dominant orientation must follow the grating angle (paper convention)."""
    y, x = np.mgrid[0:128, 0:160].astype(np.float32)
    for ang in (0.0, 0.4, 1.1, -0.7):
        img = (127 + 100 * np.cos(0.35 * (x * np.cos(ang) + y * np.sin(ang)))).astype(np.float32)
        f = cb.SteerableFiltersG2(img)
        o = ref.SteerableFiltersG2(img)
        c = (slice(20, -20), slice(20, -20))
        assert_angle_close(f.theta[c], o.theta[c], o.strength[c], np.pi, f"grating{ang}", thresh_frac=0.1)


def test_setup_is_recallable_and_getters_track():
    a, b = synth(1, 60, 70), synth(2, 33, 45)
    f = cb.SteerableFiltersG2(a)
    first = f.g2a.copy()
    f.setup(b)
    assert f.g2a.shape == (33, 45)
    f.setup(a)
    assert np.array_equal(f.g2a, first)


def test_point_overloads():
    img = synth(11, 50, 60)
    f = cb.SteerableFiltersG2(img)
    o = ref.SteerableFiltersG2(img)
    rng = basis_range([getattr(o, k) for k in STATE])
    for (x, y, th) in ((0, 0, 0.2), (59, 49, -1.0), (30, 25, 2.2)):
        got = f.steer(th, point=(x, y))
        want = o.steer_point((x, y), th, full=True)
        for i, tol in enumerate((rng, rng, float(o.c1.max() - o.c1.min()), rng)):   # e: 1e-4 of c1's own range
            assert abs(float(got[i]) - float(want[i])) <= 1e-4 * tol
        assert abs(float(got[4]) - float(want[4])) <= 1e-3 or float(want[3]) < 1e-3 * rng
        g2, h2 = f.steer(th, full=False, point=(x, y))
        assert g2 == got[0] and h2 == got[1]


def test_pointwise_statics_vs_oracle():
    rs = np.random.default_rng(3)
    g = rs.normal(0, 50, (37, 41)).astype(np.float32)
    h = rs.normal(0, 50, (37, 41)).astype(np.float32)
    g[0, 0] = h[0, 0] = 0
    g[0, 1], h[0, 1] = -3.0, 0.0
    f = cb.SteerableFiltersG2(g)
    mag, ph = f.computeMagnitudeAndPhase(g, h)
    wm, wp = ref.compute_magnitude_and_phase(g, h)
    assert np.max(np.abs(mag - wm)) <= 1e-4 * 50
    assert float(np.max(np.abs(ph - wp))) <= 2e-6          # same polynomial atan: near bit-exact
    for phi, sg in ((np.pi / 2, False), (0.0, True), (np.pi, True), (1.0, True), (-2.0, False)):
        lam = cb.SteerableFiltersG2.phaseWeights(wp, phi, sg, 2.0)
        assert float(np.max(np.abs(lam - ref.phase_weights(wp, phi, sg)))) <= 1e-5, (phi, sg)
    for fn_g, fn_o in ((f.findEdges, ref.find_edges), (f.findDarkLines, ref.find_dark_lines),
                       (f.findBrightLines, ref.find_bright_lines)):
        assert float(np.max(np.abs(fn_g(wm, wp) - fn_o(wm, wp)))) <= 1e-4 * float(wm.max())


def test_errors():
    with pytest.raises(capi.CvsError) as e:
        cb.SteerableFiltersG2(np.zeros((0, 5), np.float32))
    assert e.value.code == capi.ERR_INVALID_ARG
    with pytest.raises(capi.CvsError):
        cb.SteerableFiltersG2(synth(1, 8, 8), width=0)
    with pytest.raises(capi.CvsError):
        cb.SteerableFiltersG2(synth(1, 8, 8), width=40)
    f = cb.SteerableFiltersG2(synth(1, 8, 9))
    with pytest.raises(capi.CvsError) as e:
        f.steer(np.zeros((8, 8), np.float32))
    assert e.value.code == capi.ERR_SIZE_MISMATCH
    with pytest.raises(capi.CvsError):
        f.steer(0.1, point=(9, 0))


@pytest.mark.parametrize("width,spacing", [(3, 0.8), (5, 0.55), (7, 0.4), (1, 1.0), (12, 0.25)])
def test_generic_width_path(width, spacing):
    img = synth(31 + width, 70, 90)
    o = ref.SteerableFiltersG2(img, width, spacing)
    f = cb.SteerableFiltersG2(img, width, spacing)
    rng = _check_state(f, o, f"w{width}:")
    th = f.getDominantOrientationAngle()
    _check_steer(f.steer(th), o, th, rng, f"w{width}:")


def test_width4_other_spacing_uses_march_path():
    img = synth(41, 90, 140)
    o = ref.SteerableFiltersG2(img, 4, 0.5)
    f = cb.SteerableFiltersG2(img, 4, 0.5)
    _check_state(f, o, "s0.5:")
