"""Generate tests/golden/* from the reference's own test fixtures.

    python tests/golden/make_golden.py [--reference <headupinclouds/cvsteer checkout>]

With --reference, fish_fixture.npz is rebuilt from the reference's test data (read-only,
reference test/test.cpp:41-44):
    test/Pterois_volitans_Manado-e_edit_smallest.h   input JPEG (256x185 gray)
    test/edges.h, test/linesDark.h, test/linesBright.h   expected-output JPEGs
The `xxd -i` byte arrays are parsed as text, the JPEG bytes decoded with cv2
(IMREAD_GRAYSCALE, as test/test.cpp:53-56 does) and the DECODED PIXELS are stored,
so the fixtures do not depend on the libjpeg build of whichever machine runs the tests.
Without it, the committed fish_fixture.npz is used.

Then the float-level oracle outputs on the fish image (cv2 4.13.0) are recorded in
fish_oracle_cv2_4_13.json as regression vectors for the oracle itself and as GPU parity
fixtures: per plane its shape, the SHA-256 of its float32 bytes and the values at 32 seeded
positions (the planes themselves, 6.5 MB, are rebuilt by the oracle at test time and checked
against these bit for bit); and the default taps in taps_default.npz.
"""
import argparse
import json
import os
import re
import sys

import cv2
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", ".."))
from oracle import cvsteer_ref as ref  # noqa: E402
from tests.util import fish_oracle_planes, plane_digest  # noqa: E402

SAMPLES = 32


def read_xxd(path):
    txt = open(path).read()
    data = bytes(int(h, 16) for h in re.findall(r"0x([0-9a-fA-F]{2})", txt))
    n = int(re.search(r"_len\s*=\s*(\d+)\s*;", txt).group(1))
    assert len(data) == n, (path, len(data), n)
    return data


def decode(path):
    img = cv2.imdecode(np.frombuffer(read_xxd(path), np.uint8), cv2.IMREAD_GRAYSCALE)
    assert img is not None and img.ndim == 2
    return img


def write_fixture(reference):
    t = os.path.join(reference, "test")
    fish = decode(f"{t}/Pterois_volitans_Manado-e_edit_smallest.h")
    edges = decode(f"{t}/edges.h")
    dark = decode(f"{t}/linesDark.h")
    bright = decode(f"{t}/linesBright.h")
    assert fish.shape == (185, 256) and int(fish.sum()) == 6968201, (fish.shape, fish.sum())
    np.savez_compressed(os.path.join(HERE, "fish_fixture.npz"), fish=fish, edges_gt=edges,
                        lines_dark_gt=dark, lines_bright_gt=bright)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reference", help="headupinclouds/cvsteer checkout: rebuild fish_fixture.npz from its test data")
    a = ap.parse_args()
    if a.reference:
        write_fixture(a.reference)
    fish = np.load(os.path.join(HERE, "fish_fixture.npz"))["fish"]

    # float-level oracle outputs (cv2 4.13.0) on the fish image: digest + seeded sample per plane, one plane per line
    out = {k: np.ascontiguousarray(v, np.float32) for k, v in fish_oracle_planes(fish).items()}
    lines = []
    for k, v in out.items():
        idx = np.sort(np.random.default_rng(0).choice(v.size, min(SAMPLES, v.size), replace=False))
        entry = {"shape": list(v.shape), "sha256": plane_digest(v), "sample_index": [int(i) for i in idx],
                 "sample": [float(x) for x in v.reshape(-1)[idx]]}
        lines.append(f"  {json.dumps(k)}: {json.dumps(entry)}")
    with open(os.path.join(HERE, "fish_oracle_cv2_4_13.json"), "w") as f:
        f.write('{"cv2": %s,\n "input": "fish_fixture.npz fish (uint8 185x256), width 4 spacing 0.67 (G2/H2), '
                'width 6 spacing 0.5 (G4/H4)",\n "planes": {\n%s\n }\n}\n' % (json.dumps(cv2.__version__), ",\n".join(lines)))

    f2, f4 = ref.SteerableFiltersG2(fish), ref.SteerableFiltersG4(fish)
    taps = {n: getattr(f2, n)[0] for n in ("g1", "g2", "g3", "h1", "h2", "h3", "h4")}
    taps.update({"G4_" + n: getattr(f4, n)[0] for n in
                 ("g1", "g2", "g3", "g4", "g5", "h1", "h2", "h3", "h4", "h5", "h6")})
    np.savez(os.path.join(HERE, "taps_default.npz"), **taps)
    print("wrote fixtures; cv2", cv2.__version__)


if __name__ == "__main__":
    main()
