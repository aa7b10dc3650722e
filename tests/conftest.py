import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def fish_fixture():
    return dict(np.load(os.path.join(GOLDEN, "fish_fixture.npz")))


@pytest.fixture(scope="session")
def fish_oracle_golden():
    """Per plane of the oracle on the fish image: shape, SHA-256 and a seeded sample of the committed cv2 4.13.0 vectors."""
    import json
    with open(os.path.join(GOLDEN, "fish_oracle_cv2_4_13.json")) as f:
        return json.load(f)["planes"]


@pytest.fixture(scope="session")
def fish_oracle(fish_fixture, fish_oracle_golden):
    """The committed cv2 4.13.0 vectors in full: rebuilt by the oracle and checked bit for bit against their digests."""
    from tests import util
    planes = util.fish_oracle_planes(fish_fixture["fish"])
    assert sorted(planes) == sorted(fish_oracle_golden)
    for k, v in planes.items():
        util.assert_matches_golden(k, v, fish_oracle_golden[k])
    return planes


@pytest.fixture(scope="session")
def taps_default():
    return dict(np.load(os.path.join(GOLDEN, "taps_default.npz")))


def pytest_sessionfinish(session, exitstatus):
    """Achieved parity errors per compared quantity (max over every comparison of the session) -> gpurun_out/parity_achieved.json."""
    try:
        import json
        from tests import util
        if not util.RECORDS:
            return
        import re
        agg = {}
        for r in util.RECORDS:
            key = r["kind"] + ":" + re.sub(r"\s+", " ", re.sub(r"[-+]?\d[\d.e+-]*|\(.*?\)", "#", r["name"])).strip()
            a = agg.setdefault(key, {"max_err": 0.0, "tol_at_max": r["tol"], "worst_err_over_tol": 0.0, "comparisons": 0, "elements": 0})
            a["comparisons"] += 1
            a["elements"] += r["n"]
            ratio = r["err"] / r["tol"] if r["tol"] > 0 else (0.0 if r["err"] == 0 else float("inf"))
            if ratio >= a["worst_err_over_tol"]:
                a["worst_err_over_tol"], a["max_err"], a["tol_at_max"] = ratio, r["err"], r["tol"]
        os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
        with open(os.path.join(ROOT, "gpurun_out", "parity_achieved.json"), "w") as f:
            json.dump({"note": "range: max abs error vs rtol x range (basis planes: 1e-4 of the basis range; quadratic planes c1..c3 / "
                               "strength / e: 1e-4 of the plane's OWN range); angle: max circular error in rad where strength or "
                               "magnitude exceeds the stated fraction of its maximum",
                       "quantities": dict(sorted(agg.items()))}, f, indent=1)
    except Exception:   # reporting must never fail the run
        pass
