"""Record golden_yuv.npz: a few small cv.cvtColor results between BGR and YUV 4:2:0, so that machines without cv2 can
check the conversions.  Run with cv2 installed: python tests/golden/gen_golden_yuv.py"""
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))


def cases():
    """(name, kind, input) with kind "nv12" / "i420" (YUV -> BGR) or "bgr" (BGR -> I420)."""
    rng = np.random.default_rng(2026)
    out = []
    for w, h in ((2, 2), (8, 6), (34, 18)):
        for fmt in ("nv12", "i420"):
            out.append((f"{fmt}_{w}x{h}", fmt, rng.integers(0, 256, (h * 3 // 2, w), dtype=np.uint8)))
    for w, h in ((2, 2), (10, 6), (64, 40)):
        out.append((f"bgr_{w}x{h}", "bgr", rng.integers(0, 256, (h, w, 3), dtype=np.uint8)))
    corners = np.array([[b, g, r] for b in (0, 255) for g in (0, 255) for r in (0, 255)], np.uint8)
    out.append(("bgr_corners", "bgr", np.repeat(np.repeat(corners.reshape(2, 4, 3), 2, 0), 2, 1)))
    low = np.zeros((4, 32), np.uint8)  # Y < 16 and extreme chroma
    low[:2] = np.arange(32, dtype=np.uint8) // 2
    low[2:] = np.array([0, 255] * 16, np.uint8)
    for fmt in ("nv12", "i420"):
        out.append((f"{fmt}_low_luma", fmt, np.concatenate([low[:2], low[:2], low[2:]], 0)[:6]))
    return out


def main():
    import cv2 as cv

    codes = {"nv12": cv.COLOR_YUV2BGR_NV12, "i420": cv.COLOR_YUV2BGR_I420, "bgr": cv.COLOR_BGR2YUV_I420}
    data = {}
    for name, kind, x in cases():
        data[name + "__in"] = x
        data[name + "__out"] = cv.cvtColor(x, codes[kind])
    np.savez_compressed(os.path.join(HERE, "golden_yuv.npz"), **data)
    print(f"{len(data) // 2} cases, cv2 {cv.__version__}")


if __name__ == "__main__":
    main()
