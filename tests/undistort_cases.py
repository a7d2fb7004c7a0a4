"""Cameras, sizes and images shared by the UNDISTORTED_IMAGE tests (tests/test_undistort_host.py, tests/test_gpu_undistort.py) and
by tests/golden/make_undistort_golden.py."""
import numpy as np

K_640 = (811.4, 811.5, 307.4, 248.9)          # (fx, fy, cx, cy) of a 640x480 camera
# OpenCV's (k1, k2, p1, p2[, k3])
CAMERAS = {
    "zero": (0.0, 0.0, 0.0, 0.0),
    "barrel": (-0.35, 0.12, 0.001, -0.0007),
    "pincushion": (0.25, 0.08, 0.0, 0.0),
    "tangential": (0.0, 0.0, 0.004, -0.003),
    "k3": (0.1, -0.05, 0.0005, 0.0002, 0.02),
    # maps far outside the image: source coordinates saturate int16 (and 32 * u saturates int32)
    "extreme": (1e3, 1e5, 0.5, -0.5, 1e8),
}
SIZES = ((480, 640), (720, 1280), (479, 641), (8, 8))          # (height, width)


def camera_K(H, W):
    """K_640 scaled to a W-wide image, principal point scaled with the size"""
    s = W / 640.0
    return np.array([K_640[0] * s, K_640[1] * s, K_640[2] * s, K_640[3] * H / 480.0], np.float32)


def images(H, W, seed=0):
    """random, blurred random, all 0 and all 255"""
    from scipy.ndimage import gaussian_filter
    rng = np.random.default_rng(seed)
    rand = rng.integers(0, 256, (H, W), dtype=np.uint8)
    blur = np.clip(np.rint(gaussian_filter(rng.integers(0, 256, (H, W)).astype(np.float64), 2.0) * 1.8 - 100), 0, 255).astype(np.uint8)
    return {"random": rand, "blurred": blur, "zeros": np.zeros((H, W), np.uint8), "full": np.full((H, W), 255, np.uint8)}


def assert_maps_match(ours, cv, what=""):
    """Maps against OpenCV's: bit-exact except (a) entries within 1e-9 px of zero (cv2 leaves a rounding residue there for kc = 0)
    and (b) a few entries one float ulp apart where the distortion terms cancel (cv2's vectorised loop rounds differently there). Both
    round to the same 1/32 px, so remapped images are identical."""
    diff = ours != cv
    tiny = diff & (np.abs(cv) < 1e-9)
    ulp = diff & ~tiny & (np.abs(ours.astype(np.float64) - cv) <= np.abs(np.spacing(cv)))
    assert not (diff & ~tiny & ~ulp).any(), (what, np.argwhere(diff & ~tiny & ~ulp)[:5])
    assert ulp.sum() <= max(4, 2e-5 * ours.size), (what, int(ulp.sum()))
