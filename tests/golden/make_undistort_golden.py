"""Writes tests/golden/undistort_golden.npz with OpenCV: cv2.initUndistortRectifyMap(K, kc, None, K, size, CV_32FC1) and
cv2.remap(INTER_LINEAR, BORDER_CONSTANT, 0) — the two calls of moped's UNDISTORTED_IMAGE step — for every camera of
tests/undistort_cases.py:

    <camera>/<H>x<W>/{K, kc, mx, my, img, out}     whole maps and images at 60x80 and 8x8
    <camera>/479x641/{K, kc, rows, mx, my}         rows 0, 1, 239 and 478 of the maps of an odd-sized 641x479 image

K and kc are the float32 values the C ABI takes, widened to double for cv2. cv2.__version__ is stored under "cv2_version".

    python tests/golden/make_undistort_golden.py
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))


def main():
    import cv2
    from undistort_cases import CAMERAS, camera_K, images
    out = {"cv2_version": np.array(cv2.__version__)}
    for name, kc in CAMERAS.items():
        kc32 = np.asarray(kc, np.float32)
        for H, W in ((60, 80), (8, 8), (479, 641)):
            K = camera_K(H, W)
            A = np.array([[K[0], 0, K[2]], [0, K[1], K[3]], [0, 0, 1]], np.float64)
            mx, my = cv2.initUndistortRectifyMap(A, kc32.astype(np.float64), None, A, (W, H), cv2.CV_32FC1)
            key = f"{name}/{H}x{W}"
            out[key + "/K"], out[key + "/kc"] = K, kc32
            if H == 479:
                rows = np.array([0, 1, 239, 478])
                out[key + "/rows"], out[key + "/mx"], out[key + "/my"] = rows, mx[rows], my[rows]
                continue
            img = images(H, W, seed=7)["blurred"]
            out[key + "/mx"], out[key + "/my"], out[key + "/img"] = mx, my, img
            out[key + "/out"] = cv2.remap(img, mx, my, cv2.INTER_LINEAR, borderMode=cv2.BORDER_CONSTANT, borderValue=0)
    path = os.path.join(HERE, "undistort_golden.npz")
    np.savez_compressed(path, **out)
    print(path, os.path.getsize(path), "bytes, cv2", cv2.__version__)


if __name__ == "__main__":
    main()
