"""Writes tests/golden/nv12_rgb.npz: NV12 frames and what OpenCV's cvtColor(COLOR_YUV2RGB_NV12) makes of them, the
reference for the NV12 rule of the frame-descriptor entries (tests/test_frame_src_host.py).

    python tests/golden/make_nv12_golden.py       (needs cv2)

Small frames of seeded random bytes are stored whole: uniform bytes put Y at both ends (<= 16, >= 235) and U and V at
0 and 255.  The 1920x1080 frame is a pattern that needs no generator (nv12_pattern): its U,V pairs run through all
65536 combinations and Y through all 256 values, and only the SHA-256 of its RGB output is stored."""
import hashlib
from pathlib import Path

import numpy as np

SMALL = [(2, 2), (64, 48), (130, 98)]


def nv12_pattern(w: int, h: int) -> np.ndarray:
    """a [h*3/2][w] NV12 frame: Y = (x + 3y) mod 256, U,V pair k = row-major index of the pair: U = k mod 256,
    V = (k div 256) mod 256"""
    y = ((np.arange(w)[None, :] + 3 * np.arange(h)[:, None]) % 256).astype(np.uint8)
    k = np.arange((h // 2) * (w // 2)).reshape(h // 2, w // 2)
    uv = np.stack([k % 256, (k // 256) % 256], -1).astype(np.uint8).reshape(h // 2, w)
    return np.concatenate([y, uv], 0)


def main():
    import cv2
    rng = np.random.default_rng(2024)
    out = {"opencv_version": np.array(cv2.__version__)}
    for w, h in SMALL:
        nv12 = rng.integers(0, 256, (h * 3 // 2, w), dtype=np.uint8)
        out[f"nv12_{w}x{h}"] = nv12
        out[f"rgb_{w}x{h}"] = cv2.cvtColor(nv12, cv2.COLOR_YUV2RGB_NV12)
    rgb = cv2.cvtColor(nv12_pattern(1920, 1080), cv2.COLOR_YUV2RGB_NV12)
    out["pattern_1920x1080_sha256"] = np.array(hashlib.sha256(np.ascontiguousarray(rgb).tobytes()).hexdigest())
    np.savez_compressed(Path(__file__).resolve().parent / "nv12_rgb.npz", **out)


if __name__ == "__main__":
    main()
