"""Generates tests/golden/qt6/qt6_raster.npz: what the real Qt 6.6.3 raster engine (the libraries that ship
with Nsight Compute, linked into oracle/_ref/libenv_ref_qt6.so by oracle/build_ref.py --qt6) draws for
every case of the Qt 6 tests in tests/test_oracle.py. Needs those libraries; the tests do not.
  python tests/golden/qt6/make_qt6_golden.py
Frame cases: <key>_digest = 64-bit digest of Qt's rgb batch after each step, <key>_patch = rows
(step, env, y, x, r, g, b) of the pixels in which Qt differs from the CPU raster restatement.
Draw sweeps: <key>_digest = 64-bit digest of Qt's image for each draw, in the order the tests draw."""
import ctypes as C
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
TESTS = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(TESTS))
sys.path.insert(0, TESTS)
from oracle import build_ref, qt6_support  # noqa: E402
from oracle.ref_env import REF_LIB, REF_LIB_QT6  # noqa: E402
from test_oracle import (QT6_FRAME_CASES, digest64, ellipse_and_line_draws, qt6_case_frames,  # noqa: E402
                         scaled_blit_and_fill_draws)


def main():
    if not qt6_support.available():
        raise SystemExit("Qt 6 libraries (Nsight Compute) not found")
    if not (os.path.exists(REF_LIB) and os.path.exists(REF_LIB_QT6)):
        build_ref.build(qt6=True)
    out = {}
    for key in QT6_FRAME_CASES:
        digests, patch = [], []
        for t, (mine, qt) in enumerate(zip(qt6_case_frames(key), qt6_case_frames(key, REF_LIB_QT6))):
            digests.append(digest64(qt))
            for e, y, x in np.argwhere((mine != qt).any(-1)):
                patch.append((t, e, y, x, *qt[e, y, x]))
        out[key + "_digest"] = np.array(digests, np.uint64)
        out[key + "_patch"] = np.array(patch, np.int32).reshape(-1, 7)
        print(key, len(digests), "steps,", len(patch), "pixels differ")
    qt = C.CDLL(REF_LIB_QT6, handle=qt6_support.lazy_dlopen(REF_LIB_QT6))
    for key, draws in (("ellipse_line", ellipse_and_line_draws), ("blit_fill", scaled_blit_and_fill_draws)):
        out[key + "_digest"] = np.array([digest64(img) for _, img in draws(qt)], np.uint64)
        print(key, len(out[key + "_digest"]), "draws")
    np.savez_compressed(os.path.join(HERE, "qt6_raster.npz"), **out)


if __name__ == "__main__":
    main()
