"""Generate the committed golden vectors from the UNMODIFIED reference.

Runs only in the build container, where /root/reference (OpenStitching/stitching v0.7.0) and its numeric
backend cv2 4.13.0 are importable:

    python tests/golden/gen_golden.py

Every expected output below is produced by the reference's own classes
(stitching.warper.Warper, stitching.blender.Blender -- reference files stitching/warper.py, stitching/blender.py)
or, for the pyramid primitives, by the cv2 calls OpenCV's blender makes internally.  The fixtures are replayed by
tests/test_oracle_golden.py (CPU oracle) and tests/test_gpu_parity.py (CUDA path); neither needs the reference.
"""
import hashlib
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", ".."))
sys.path.insert(0, os.path.join(HERE, ".."))
sys.path.insert(0, "/root/reference")

import cv2 as cv  # noqa: E402
from stitching.blender import Blender as RefBlender  # noqa: E402
from stitching.warper import Warper as RefWarper  # noqa: E402

import replay  # noqa: E402
from stitching_b200 import rigs  # noqa: E402


def rot(rx, ry, rz):
    cz, sz = np.cos(rz), np.sin(rz)
    Rz = np.array([[cz, -sz, 0], [sz, cz, 0], [0, 0, 1]])
    return (Rz @ rigs.rot_y(ry) @ rigs.rot_x(rx)).astype(np.float32)


def gen_warp():
    rng = np.random.default_rng(20260922)
    cases = []
    W, H = 96, 72
    specs = [
        ("spherical", rot(0.05, 0.3, 0.02), 90.0, 80.0),
        ("spherical", rot(1.35, -2.9, 0.1), 70.0, 75.0),     # pole in view, +-pi wrap
        ("spherical", rot(-1.5, 1.0, -0.2), 60.0, 60.0),     # other pole
        ("spherical", rot(0.2, 3.1, 0.0), 120.0, 100.0),     # z <= 0 region / wrap
        ("cylindrical", rot(0.1, -0.4, 0.05), 90.0, 100.0),
        ("cylindrical", rot(-0.3, 2.8, 0.2), 75.0, 60.0),
        ("cylindrical", rot(0.4, -3.0, -0.1), 110.0, 95.0),
        ("plane", rot(0.05, 0.1, 0.02), 90.0, 90.0),
        ("plane", rot(0.4, -0.7, 0.3), 80.0, 60.0),          # steep: far out-of-range coordinates
        ("plane", rot(-0.2, 0.9, -0.1), 100.0, 140.0),
    ]
    for k, (wtype, R, focal, scale) in enumerate(specs):
        cam = rigs.Camera(focal, 1.0 + 0.03 * (k % 3 - 1), W / 2 + 3.5 * (k % 2), H / 2 - 2.25, R)
        cases.append((wtype, cam, scale, 1.0))
    # the other twelve names of warper.py:10-27 (two cameras each; tests/test_stitcher.py:85,110 of the reference use
    # fisheye and compressedPlaneA2B1)
    extra = ["fisheye", "stereographic", "compressedPlaneA2B1", "compressedPlaneA1.5B1", "compressedPlanePortraitA2B1",
             "compressedPlanePortraitA1.5B1", "paniniA2B1", "paniniA1.5B1", "paniniPortraitA2B1", "paniniPortraitA1.5B1", "mercator",
             "transverseMercator"]
    for k, wtype in enumerate(extra):
        cases.append((wtype, rigs.Camera(95.0 + 3 * k, 1.0 + 0.02 * (k % 3 - 1), W / 2 + 2.5 * (k % 2), H / 2 - 1.25, rot(0.04 * (k % 4), 0.25 - 0.05 * k, 0.02)),
                      88.0 + 2 * k, 1.0))
        cases.append((wtype, rigs.Camera(70.0 + 2 * k, 1.0, W / 2, H / 2, rot(-0.3 + 0.03 * k, -0.45 + 0.06 * k, 0.15)), 64.0 + 3 * k,
                      [1.0, 0.8][k % 2]))
    for k in range(3):
        th, s = [0.03, -0.2, 0.11][k], [1.0, 0.9, 1.15][k]
        Hm = np.array([[s * np.cos(th), -s * np.sin(th), [12.5, -80.25, 301.0][k]],
                       [s * np.sin(th), s * np.cos(th), [-7.75, 40.0, -33.5][k]], [0, 0, 1]], np.float32)
        cases.append(("affine", rigs.Camera(1.0, 1.0, 0.0, 0.0, Hm), 1.0, [1.0, 1.0, 0.75][k]))
    out = {"n": len(cases)}
    src_sha = hashlib.sha256()  # the sources are drawn again from the seed (replay.warp_cases), not stored
    for i, (wtype, cam, scale, aspect) in enumerate(cases):
        img = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
        wr = RefWarper(wtype)
        wr.scale = scale
        out[f"type_{i}"] = wtype
        out[f"cam_{i}"] = np.array([cam.focal, cam.aspect, cam.ppx, cam.ppy], np.float64)
        out[f"R_{i}"] = cam.R
        out[f"scale_{i}"] = np.float64(scale)
        out[f"aspect_{i}"] = np.float64(aspect)
        src_sha.update(img.tobytes())
        out[f"roi_{i}"] = np.array(wr.warp_roi((W, H), cam, aspect), np.int64)
        replay.pack(out, f"img_{i}", wr.warp_image(img, cam, aspect))
        replay.pack(out, f"mask_{i}", wr.create_and_warp_mask((W, H), cam, aspect))
    out["src_sha256"] = src_sha.hexdigest()
    np.savez_compressed(os.path.join(HERE, "golden_warp.npz"), **out)
    print("warp cases", len(cases))


def make_mask(kind, h, w, rng):
    if kind == "full":
        return np.full((h, w), 255, np.uint8)
    if kind == "box":
        m = np.zeros((h, w), np.uint8)
        m[h // 5: h - h // 6, w // 7: w - w // 5] = 255
        return m
    if kind == "speckle":
        return (rng.random((h, w)) > 0.3).astype(np.uint8) * 255
    if kind == "ramp":
        return np.clip(np.add.outer(np.arange(h), np.arange(w)) * 3, 0, 255).astype(np.uint8)
    if kind == "gray":
        return rng.integers(0, 256, (h, w), dtype=np.uint8)
    raise KeyError(kind)


def gen_blend():
    rng = np.random.default_rng(7)
    specs = [  # (blender, strength, mask kind, n images, int16 feed)
        ("multiband", 5, "full", 3, False),
        ("multiband", 5, "ramp", 3, False),
        ("multiband", 20, "gray", 2, False),
        ("multiband", 60, "box", 3, False),
        ("multiband", 100, "speckle", 2, False),   # nb clipped by ceil(log2(max(w,h)))
        ("multiband", 2, "full", 2, False),        # 0 bands
        ("multiband", 20, "ramp", 2, True),        # generic int16 input incl. negatives
        ("feather", 5, "box", 3, False),
        ("feather", 20, "speckle", 2, False),
        ("feather", 5, "full", 2, True),
        ("no", 5, "gray", 3, False),
        ("multiband", 0.2, "box", 2, False),       # blend width < 1 -> NO blender
    ]
    out = {"n": len(specs)}
    for i, (btype, strength, mk, n, s16) in enumerate(specs):
        imgs, masks, corners = [], [], []
        for j in range(n):
            w, h = int(rng.integers(40, 110)), int(rng.integers(30, 90))
            img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8) if (i + j) % 2 else rigs.synth_image(h, w, 50 + 10 * i + j)
            if s16:
                img = img.astype(np.int16) * 3 - 150
            imgs.append(img)
            masks.append(make_mask(mk, h, w, rng))
            corners.append((int(rng.integers(-60, 60)), int(rng.integers(-40, 40))))
        sizes = [(m.shape[1], m.shape[0]) for m in masks]
        b = RefBlender(btype, strength)
        b.prepare(corners, sizes)
        for img, m, c in zip(imgs, masks, corners):
            b.feed(img, m, c)
        pano, pmask = b.blend()
        out[f"type_{i}"] = btype
        out[f"strength_{i}"] = np.float64(strength)
        out[f"count_{i}"] = n
        for j in range(n):
            out[f"img_{i}_{j}"] = imgs[j]
            out[f"mask_{i}_{j}"] = masks[j]
            out[f"corner_{i}_{j}"] = np.array(corners[j], np.int64)
        out[f"pano_{i}"] = pano
        out[f"pmask_{i}"] = pmask
    np.savez_compressed(os.path.join(HERE, "golden_blend.npz"), **out)
    print("blend cases", len(specs))


def gen_pyr():
    rng = np.random.default_rng(11)
    out = {}
    shapes = [(64, 96), (34, 50), (2, 2), (6, 4), (16, 2), (2, 8), (40, 136)]
    out["n"] = len(shapes)
    for i, (h, w) in enumerate(shapes):
        a = rng.integers(-3000, 3000, (h, w, 3)).astype(np.int16)
        f = rng.random((h, w), dtype=np.float32)
        out[f"s16_{i}"] = a
        out[f"f32_{i}"] = f
        out[f"down_s16_{i}"] = cv.pyrDown(a)
        out[f"down_f32_{i}"] = cv.pyrDown(f)
        out[f"up_s16_{i}"] = cv.pyrUp(a)
    v = np.array([-3, 260, -300, 100, -32768, 32767, 0, 255, -255, 256], np.int16)
    out["csa_in"] = v
    out["csa_out"] = cv.convertScaleAbs(v.reshape(1, -1)).reshape(-1)
    m = (rng.random((40, 60)) > 0.2).astype(np.uint8) * 255
    out["dt_mask"] = m
    out["dt_l1"] = cv.distanceTransform(m, cv.DIST_L1, 3)
    np.savez_compressed(os.path.join(HERE, "golden_pyr.npz"), **out)
    print("pyr cases", len(shapes))


def gen_e2e():
    """Reference Warper + Blender driven like stitcher.py:178-189, 241-259 on scaled-down BASELINE rigs."""
    out = {}
    for name, sd, ncap in (("cfg2", 20, None), ("cfg3", 20, 6), ("cfg5", 10, None)):
        cfg = rigs.config(name, sd)
        cams = cfg["cameras"][:ncap] if ncap else cfg["cameras"]
        imgs = [rigs.synth_image(cfg["h"], cfg["w"], i) for i in range(len(cams))]
        wr = RefWarper(cfg["warper"])
        wr.set_scale(cams)
        sizes_in = [(cfg["w"], cfg["h"])] * len(cams)
        warped = list(wr.warp_images(imgs, cams))
        masks = list(wr.create_and_warp_masks(sizes_in, cams))
        corners, sizes = wr.warp_rois(sizes_in, cams)
        b = RefBlender(cfg["blender"], cfg["strength"])
        b.prepare(corners, sizes)
        for img, m, c in zip(warped, masks, corners):
            b.feed(img, m, c)
        pano, pmask = b.blend()
        h = hashlib.sha256()
        for im in imgs:
            h.update(im.tobytes())
        out[f"{name}_scale_down"] = sd
        out[f"{name}_n"] = len(cams)
        out[f"{name}_input_sha256"] = h.hexdigest()
        out[f"{name}_corners"] = np.array(corners, np.int64)
        out[f"{name}_sizes"] = np.array(sizes, np.int64)
        replay.pack(out, f"{name}_pano", pano)
        replay.pack(out, f"{name}_pmask", pmask)
        print(name, "pano", pano.shape)
    np.savez_compressed(os.path.join(HERE, "golden_e2e.npz"), **out)


def gen_seam():
    """SeamFinder.resize (stitching/seam_finder.py:38-43) of the unmodified reference, fed the way stitcher.py:223-225
    feeds it: a LOW-resolution seam mask as cv.UMat and the FINAL-resolution warped mask as ndarray."""
    from stitching.seam_finder import SeamFinder as RefSeamFinder

    rng = np.random.default_rng(20260923)
    out = {}
    # warped validity masks of a scaled cfg2 rig at "final" resolution; seam masks at ~1/3 of it, like 0.1 vs 1 MP
    cfg = rigs.config("cfg2", 10)
    cams = cfg["cameras"][:4]
    wr = RefWarper(cfg["warper"])
    wr.set_scale(cams)
    masks = list(wr.create_and_warp_masks([(cfg["w"], cfg["h"])] * len(cams), cams))
    cases = []
    for i, m in enumerate(masks):
        h, w = m.shape
        sh, sw = int(round(h / 3.17)) + i, int(round(w / 3.17)) - i  # the two resolutions round independently
        seam = np.zeros((sh, sw), np.uint8)
        seam[:, : sw // 2 + int(rng.integers(-5, 6))] = 255  # a seam through the middle ...
        for _ in range(6):  # ... with a ragged edge
            cv.circle(seam, (sw // 2, int(rng.integers(0, sh))), int(rng.integers(2, 9)), int(rng.integers(0, 2)) * 255, -1)
        cases.append((seam, m))
    cases.append(((rng.random((37, 53)) < 0.5).astype(np.uint8) * 255, np.full((371, 533), 255, np.uint8)))  # noise, 10x
    cases.append((rng.integers(0, 256, (40, 30), dtype=np.uint8), (rng.random((97, 61)) < 0.8).astype(np.uint8) * 255))  # gray levels
    cases.append((rng.integers(0, 256, (64, 48), dtype=np.uint8), np.full((32, 24), 255, np.uint8)))  # exact 2x reduction
    cases.append((rng.integers(0, 256, (50, 70), dtype=np.uint8), np.full((31, 45), 255, np.uint8)))  # other reduction
    cases.append((np.array([[255]], np.uint8), np.full((5, 7), 255, np.uint8)))  # 1x1 source
    for i, (seam, m) in enumerate(cases):
        got = RefSeamFinder.resize(cv.UMat(seam), m)
        out[f"seam_{i}"] = seam
        out[f"mask_{i}"] = m
        out[f"out_{i}"] = got.get() if hasattr(got, "get") else np.asarray(got)
    out["n"] = len(cases)
    np.savez_compressed(os.path.join(HERE, "golden_seam.npz"), **out)
    print("seam cases", len(cases))


def gen_gain():
    """ExposureErrorCompensator.apply (stitching/exposure_error_compensator.py:43-45) of the unmodified reference: the
    compensator estimates its gains with its own feed() on LOW-resolution views (stitcher.py:211), apply() then runs on
    FINAL-resolution images (stitcher.py:219-221).  Stored: the gains (getMatGains), the inputs and apply()'s outputs."""
    from stitching.exposure_error_compensator import ExposureErrorCompensator as RefCompensator

    rng = np.random.default_rng(20260924)
    lh, lw = 90, 120
    base = cv.resize(rng.integers(40, 200, (8, 12, 3), dtype=np.uint8), (lw + 60, lh), interpolation=cv.INTER_CUBIC).astype(np.float32)
    low = [np.clip(base[:, 0:lw] * 0.8, 0, 255).astype(np.uint8),
           np.clip(base[:, 30:30 + lw] * 1.2 + rng.normal(0, 2, (lh, lw, 3)), 0, 255).astype(np.uint8),
           np.clip(base[:, 60:60 + lw] * np.array([1.0, 0.85, 1.25]), 0, 255).astype(np.uint8)]
    corners = [(0, 0), (30, 0), (60, 0)]
    masks = [np.full((lh, lw), 255, np.uint8)] * 3
    out = {}
    k = 0
    for name in ("gain_blocks", "channel_blocks", "gain", "channel", "no"):
        comp = RefCompensator(name, 1, 32)
        comp.feed(corners, low, masks)
        gains = [np.asarray(g) for g in comp.compensator.getMatGains()] if name != "no" else [None] * 3
        for idx in range(3):
            h, w = int(rng.integers(50, 110)), int(rng.integers(70, 150))  # small fixtures: the arithmetic is per pixel
            img = rigs.noise_image(h, w, 700 + k) if idx % 2 else rigs.synth_image(h, w, 700 + k)
            got = comp.apply(idx, (0, 0), img.copy(), np.full((h, w), 255, np.uint8))
            out[f"kind_{k}"] = name
            out[f"img_{k}"] = img
            out[f"gain_{k}"] = gains[idx] if gains[idx] is not None else np.zeros((0,), np.float32)
            out[f"out_{k}"] = got.get() if hasattr(got, "get") else np.asarray(got)
            k += 1
    out["n"] = k
    np.savez_compressed(os.path.join(HERE, "golden_gain.npz"), **out)
    print("gain cases", k)


def gen_resize():
    """Images.resize_img_by_scaler (stitching/images.py:120-123) of the unmodified reference with its own scalers
    (megapix_scaler.py): full-size views down to MEDIUM / LOW / FINAL-like resolutions, plus an upscale."""
    from stitching.images import Images as RefImages
    from stitching.megapix_scaler import MegapixDownscaler, MegapixScaler

    out = {}
    k = 0
    for (h, w, mp, up) in ((150, 200, 0.015, False), (129, 195, 0.003, False), (150, 200, 0.0075, False), (64, 48, 0.000768, False),
                           (60, 45, 0.005, True), (100, 150, -1, False)):
        img = rigs.noise_image(h, w, 800 + k) if k % 2 else rigs.synth_image(h, w, 800 + k)
        scaler = (MegapixScaler if up else MegapixDownscaler)(mp)
        scaler.set_scale_by_img_size((w, h))
        out[f"img_{k}"] = img
        out[f"size_{k}"] = np.array(scaler.get_scaled_img_size((w, h)), np.int64)
        out[f"out_{k}"] = RefImages.resize_img_by_scaler(scaler, (w, h), img)
        k += 1
    out["n"] = k
    np.savez_compressed(os.path.join(HERE, "golden_resize.npz"), **out)
    print("resize cases", k, [tuple(out[f"size_{i}"]) for i in range(k)])


def gen_timelapse():
    """Timelapser.initialize / process_frame / get_frame (stitching/timelapser.py:36-52) of the unmodified reference for
    "as_is" and "crop": warped-image-sized frames at overlapping corners (negative ones too), int16-range inputs
    included (the class converts with astype(int16) and shows |.| saturated)."""
    from stitching.timelapser import Timelapser as RefTimelapser

    rng = np.random.default_rng(4242)
    out = {}
    k = 0
    for kind in ("as_is", "crop"):
        for trial in range(3):
            n = 3 + trial
            sizes = [(int(rng.integers(20, 60)), int(rng.integers(16, 48))) for _ in range(n)]
            corners = [(int(rng.integers(-15, 15)) + 10 * i, int(rng.integers(-12, 12))) for i in range(n)]
            t = RefTimelapser(kind)
            t.initialize(corners, sizes)
            out[f"kind_{k}"] = np.array(kind)
            out[f"corners_{k}"] = np.array(corners, np.int64)
            out[f"sizes_{k}"] = np.array(sizes, np.int64)
            for i, ((w, h), c) in enumerate(zip(sizes, corners)):
                img = rigs.noise_image(h, w, 900 + 10 * k + i)
                if trial == 2:  # values a uint8 image cannot hold: exercises |.| and the saturation of get_frame
                    img = (img.astype(np.int16) * 3 - 300).astype(np.int16)
                t.process_frame(img, c)
                out[f"img_{k}_{i}"] = img
                out[f"frame_{k}_{i}"] = t.get_frame()
            k += 1
    out["n"] = k
    np.savez_compressed(os.path.join(HERE, "golden_timelapse.npz"), **out)
    print("timelapse cases", k, [out[f"frame_{i}_0"].shape for i in range(k)])


if __name__ == "__main__":
    print("cv2", cv.__version__)
    gen_warp()
    gen_blend()
    gen_pyr()
    gen_e2e()
    gen_seam()
    gen_gain()
    gen_resize()
    gen_timelapse()
    for f in sorted(os.listdir(HERE)):
        if f.endswith(".npz"):
            print(f, os.path.getsize(os.path.join(HERE, f)) // 1024, "KiB")
