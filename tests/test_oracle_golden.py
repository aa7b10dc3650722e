"""Pins the oracle (oracle/cvsteer_ref.py) against the reference's own acceptance test and
against the frozen known-answer values of SURVEY.md App. C.  CPU only."""
import cv2
import numpy as np
import pytest

from oracle import cvsteer_ref as ref
from tests.util import assert_matches_golden


def _recode(x):
    # test/test.cpp:64-69 -- JPEG encode+decode to reproduce the loss baked into the GT images
    ok, buf = cv2.imencode(".jpg", x)
    assert ok
    return cv2.imdecode(buf, cv2.IMREAD_GRAYSCALE)


def test_reference_gtest_basic(fish_fixture):
    """TEST(cvsteer, basic), test/test.cpp:70-103: mean-L1 <= 1.0 grey level on 3 maps."""
    fish = fish_fixture["fish"]
    assert fish.shape == (185, 256) and int(fish.sum()) == 6968201
    f, (g2, h2, e, mag, phase) = ref.g2_full(fish, 4, 0.67)
    # both reference callers feed `magnitude`, not `e` (test/test.cpp:88-90)
    maps = {
        "edges_gt": ref.find_edges(mag, phase),
        "lines_dark_gt": ref.find_dark_lines(mag, phase),
        "lines_bright_gt": ref.find_bright_lines(mag, phase),
    }
    for name, m in maps.items():
        out8 = ref.normalize_minmax_u8(m)
        err = cv2.norm(_recode(out8), fish_fixture[name], cv2.NORM_L1) / float(fish.size)
        assert err <= 1.0, (name, err)
        # the restatement is in fact far tighter than the reference's threshold
        assert err <= 0.05, (name, err)


# SURVEY.md App. C: (min, max, float64 sum, value at [92,128])
KNOWN = {
    "g2a": (-272.3235, 332.5981, -9882.026, -92.52432),
    "g2b": (-183.1040, 176.9852, 96.153, 30.13642),
    "g2c": (-255.7264, 261.9788, -10204.595, -2.13215),
    "h2a": (-316.2635, 314.1828, 4989.103, -12.67481),
    "h2b": (-113.6658, 113.4026, 31117.224, 1.25490),
    "h2c": (-106.4534, 103.3507, 1646.453, -0.72962),
    "h2d": (-306.5441, 276.4650, 93966.261, 42.62686),
    "g4a": (-487.7033, 446.9799, -34993.710, 153.86104),
    "g4e": (-363.2922, 326.8790, -34684.441, -8.69672),
    "h4a": (-449.9319, 493.1993, 1873.672, 18.01436),
    "h4f": (-367.3312, 328.2269, 36214.978, -38.57962),
}


def test_known_answers_fish(fish_fixture):
    fish = fish_fixture["fish"]
    f2 = ref.SteerableFiltersG2(fish)
    f4 = ref.SteerableFiltersG4(fish)
    for name, (mn, mx, sm, v) in KNOWN.items():
        p = getattr(f2 if name[1] == "2" else f4, name)
        assert p.dtype == np.float32 and p.shape == fish.shape
        assert abs(float(p.min()) - mn) < 2e-3, name
        assert abs(float(p.max()) - mx) < 2e-3, name
        # plane sums cancel heavily (|sum| ~1e4 of sum|x| ~1e6): a 1-ulp difference in one tap moves them by ~1
        assert abs(float(p.astype(np.float64).sum()) - sm) < 5.0, name
        assert abs(float(p[92, 128]) - v) < 2e-4, name
    assert abs(float(f2.theta[92, 128]) - 0.354760) < 1e-5
    assert abs(float(f2.strength[92, 128]) - 4604.653320) < 0.01
    assert abs(float(f2.c1[92, 128]) - 4358.150879) < 0.01
    assert float(f2.theta.min()) >= -np.pi / 2 - 1e-6 and float(f2.theta.max()) <= np.pi / 2 + 1e-6
    g4, h4 = f4.steer_scalar(0.3)
    assert abs(float(g4[92, 128]) - 191.86337) < 1e-3
    assert abs(float(h4[92, 128]) - 16.558273) < 1e-3


def test_known_taps():
    f = ref.create
    np.testing.assert_allclose(f(4, 0.67, ref.G21)[0, :5],
                               [0.00935593, 0.11477663, 0.3963536, -0.06010311, -0.9213], rtol=2e-6)
    np.testing.assert_allclose(f(4, 0.67, ref.G22)[0, :5],
                               [7.5984176e-04, 1.7595714e-02, 1.6602778e-01, 6.3832992e-01, 1.0], rtol=2e-6)
    np.testing.assert_allclose(f(4, 0.67, ref.G23)[0, :5],
                               [-0.00276453, -0.04801375, -0.30202875, -0.58060753, 0], rtol=2e-6, atol=1e-12)
    np.testing.assert_allclose(f(4, 0.67, ref.H21)[0, :5],
                               [-0.00981528, -0.06177995, 0.09973991, 0.7550229, 0], rtol=3e-6, atol=1e-12)
    np.testing.assert_allclose(f(4, 0.67, ref.H24)[0, :5],
                               [0.00477896, 0.05659223, 0.16953593, -0.18890913, -0.734967], rtol=3e-6)
    np.testing.assert_allclose(f(6, 0.5, ref.G41)[0, 6:],
                               [0.9345, 0.06064911, -0.57297224, -0.12311947, 0.10840111, 0.0506626, 0.00841883],
                               rtol=3e-6)
    np.testing.assert_allclose(f(6, 0.5, ref.H46)[0, 6:],
                               [-0.6638, -0.32226777, 0.12368107, 0.16718425, 0.06110463, 0.0107839, 0.00102877],
                               rtol=3e-6)
    # symmetry is exact (float(-i)*s == -(float(i)*s); the functions are exactly even/odd)
    for fn, odd in ((ref.G21, 0), (ref.G22, 0), (ref.G23, 1), (ref.H21, 1), (ref.H23, 1), (ref.H24, 0),
                    (ref.G41, 0), (ref.G43, 1), (ref.G44, 1), (ref.G45, 0), (ref.H41, 1), (ref.H43, 0),
                    (ref.H44, 1), (ref.H45, 1), (ref.H46, 0)):
        for w, s in ((4, 0.67), (6, 0.5), (9, 0.31)):
            k = f(w, s, fn)[0]
            assert np.array_equal(k, -k[::-1] if odd else k[::-1])


def test_golden_vectors_match_oracle(fish_fixture, fish_oracle_golden):
    """The committed float-level vectors are what the oracle produces today (same cv2)."""
    if cv2.__version__ != "4.13.0":
        pytest.skip("vectors were generated with cv2 4.13.0")
    fish = fish_fixture["fish"]
    f2, (g2, h2, e, mag, phase) = ref.g2_full(fish)
    for k in ref.SteerableFiltersG2.PLANES + ("c1", "c2", "c3", "theta", "strength"):
        assert_matches_golden(k, getattr(f2, k), fish_oracle_golden[k])
    assert_matches_golden("phase", phase, fish_oracle_golden["phase"])
    assert_matches_golden("magnitude", mag, fish_oracle_golden["magnitude"])


def test_wrap_and_phase_weights():
    a = np.array([[0.0, 1.0, np.pi, 3.2, 6.0]], np.float32)
    w = ref.wrap(a)
    assert w[0, 0] == 0 and w[0, 1] == 1 and w[0, 2] == np.float32(np.pi)  # compare is done in float: float(pi) is not > float(M_PI)
    assert abs(w[0, 3] - (3.2 - 2 * np.pi)) < 1e-6 and abs(w[0, 4] - (6.0 - 2 * np.pi)) < 1e-6
    ph = np.array([[0.0, np.pi / 2, -np.pi / 2, np.pi, -3.0, 0.3]], np.float32)
    lam_e = ref.phase_weights(ph, np.pi / 2, False)
    np.testing.assert_allclose(lam_e[0, :4], [0, 1, 1, 0], atol=1e-6)
    lam_d = ref.phase_weights(ph, 0.0, True)
    np.testing.assert_allclose(lam_d[0], [1, 0, 0, 0, 0, np.cos(0.3) ** 2], atol=1e-6)
    lam_b = ref.phase_weights(ph, np.pi, True)
    np.testing.assert_allclose(lam_b[0, 3], 1, atol=1e-6)
    np.testing.assert_allclose(lam_b[0, 4], np.cos(2 * np.pi - 3.0 - np.pi) ** 2, atol=1e-5)


def test_pyr_down_definition():
    rng = np.random.default_rng(5)
    img = rng.uniform(0, 255, (37, 51)).astype(np.float32)
    out = ref.pyr_down(img)
    assert out.shape == (19, 26)
    k = np.array([1, 4, 6, 4, 1], np.float64) / 16
    p = np.pad(img.astype(np.float64), 2, mode="reflect")
    rows = sum(k[i] * p[:, i:i + 51] for i in range(5))
    full = sum(k[i] * rows[i:i + 37, :] for i in range(5))
    np.testing.assert_allclose(out, full[::2, ::2], atol=1e-4)


def test_live_oracle_reproduces_committed_g2_vectors_bitwise(fish_fixture, fish_oracle_golden):
    """The G2/H2 vectors digested in tests/golden/fish_oracle_cv2_4_13.json were first written by tests/golden/make_golden.py
    with the literal float64 `double * Mat1f` round trip and the fancy-index `copyTo`; the oracle now uses a float32 multiply
    for the dyadic coefficients of G2.cpp:93-95 and np.copyto -- this pins that both are bit-identical to what was committed."""
    f, (g2, h2, e, mag, phase) = ref.g2_full(fish_fixture["fish"], 4, 0.67)
    live = dict(c1=f.c1, c2=f.c2, c3=f.c3, theta=f.theta, strength=f.strength, g2=g2, h2=h2, e=e, magnitude=mag, phase=phase)
    for k in ref.SteerableFiltersG2.PLANES:
        live[k] = getattr(f, k)
    for k, v in live.items():
        assert_matches_golden(k, v, fish_oracle_golden[k])
    # ... and the coefficient shortcut itself, including values the fish image does not reach
    m = (np.random.default_rng(5).standard_normal((64, 64)) * 1e4).astype(np.float32)
    m[0, :6] = [0.0, 1e-45, -1e-45, 3e38, 1e-38, -2e-38]
    for a in (0.5, 0.25, 0.375, 0.3125, 0.5625, 0.46875, 0.28125, 0.1875, 0.9375, 1.6875, 0.1):
        with np.errstate(over="ignore"):
            want = (a * m.astype(np.float64)).astype(np.float32)
            assert np.array_equal(ref._scale(a, m), want), a
