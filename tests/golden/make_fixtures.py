"""Generates tests/golden/testimg.npz from the reference's own test data.

Run where a checkout of the reference and OpenCV are present:
    python tests/golden/make_fixtures.py <reference checkout>
The reference ships no golden vectors for the hot path; what it does ship are the input images its
relational tests run on (data/testimg/*.jpg|png, used by tests/ut_se3aligner.cpp:58-77,
tests/ut_cuda_utils.cpp:32-59, tests/ut_sfmaligner.cpp:41-57).  We store them decoded (8-bit gray via
cv2.IMREAD_GRAYSCALE exactly as the tests load them, 16-bit depth in millimetres) together with
OpenCV outputs the reference tests compare against (Sobel scale 1/8, GaussianBlur 5x5 + pyrDown), so
that the known-answer tests run without the reference and without depending on the cv2 build of
the GPU machine.  The 25x25 box blur of ut_se3aligner.cpp is recomputed bit for bit by
tests/helpers.py:box_blur25 instead of being stored.
"""
import os
import sys

import cv2
import numpy as np

OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "testimg.npz")


def main(reference):
    src = os.path.join(reference, "data", "testimg")
    d = {}
    for name in ("1047", "1052"):
        g = cv2.imread(os.path.join(src, name + ".jpg"), cv2.IMREAD_GRAYSCALE)
        assert g is not None and g.dtype == np.uint8
        d["gray_" + name] = g
    dpt = cv2.imread(os.path.join(src, "1047.png"), cv2.IMREAD_ANYDEPTH)
    assert dpt is not None and dpt.dtype == np.uint16
    d["depth_1047_mm"] = dpt
    # what ut_cuda_utils.cpp compares against
    img = d["gray_1047"].astype(np.float32) * np.float32(1 / 255.0)  # convertTo(CV_32FC1, 1/255.0)
    d["ocv_sobel_x_1047"] = cv2.Sobel(img, cv2.CV_32F, 1, 0, ksize=3, scale=1 / 8.0)
    d["ocv_sobel_y_1047"] = cv2.Sobel(img, cv2.CV_32F, 0, 1, ksize=3, scale=1 / 8.0)
    blur = cv2.GaussianBlur(img, (5, 5), 0, 0)
    d["ocv_blurdown_1047"] = cv2.pyrDown(blur, dstsize=(img.shape[1] // 2, img.shape[0] // 2))
    # what ut_se3aligner.cpp:70-76 feeds the aligner (/255, 25x25 box blur) must match the test helper exactly
    tests = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path[:0] = [tests, os.path.dirname(tests)]
    from helpers import box_blur25
    for name in ("1047", "1052"):
        f = d["gray_" + name].astype(np.float32) * np.float32(1 / 255.0)
        assert np.array_equal(box_blur25(d["gray_" + name]), cv2.blur(f, (25, 25)))
    np.savez_compressed(OUT, **d)
    print("wrote", OUT, {k: (v.shape, str(v.dtype)) for k, v in d.items()})


if __name__ == "__main__":
    main(sys.argv[1])
