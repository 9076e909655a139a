"""The oracle and the drop-in classes against what the UNMODIFIED reference classes returned for the same random inputs.

The inputs are drawn from a fixed seed: every projection of Warper.WARP_TYPE_CHOICES (roi, warped image, warped mask), the
three blenders with gray and binary masks, the Timelapser, SeamFinder.resize, Images.resize_img_by_scaler and
ExposureErrorCompensator.apply.  What the reference returned for them is stored in tests/golden/golden_live.npz (see
replay.pack), recorded from an OpenStitching/stitching checkout and its cv2 with

    PYTHONPATH=. python tests/test_vs_reference_live.py <reference checkout> [seed]

A different seed gives fresh draws: record with it, then run this file.
"""
import importlib
import os
import sys

import numpy as np

import replay
from stitching_b200 import rigs

GOLDEN = "golden_live.npz"


def _rot(rx, ry, rz):
    cz, sz = np.cos(rz), np.sin(rz)
    Rz = np.array([[cz, -sz, 0], [sz, cz, 0], [0, 0, 1]])
    return (Rz @ rigs.rot_y(ry) @ rigs.rot_x(rx)).astype(np.float32)


def projection_cases(seed, types):
    rng = np.random.default_rng(seed)
    W, H = 88, 66
    for wtype in types:
        for trial in range(3):
            if wtype == "affine":
                th, s = rng.uniform(-0.2, 0.2), rng.uniform(0.85, 1.2)
                R = np.array([[s * np.cos(th), -s * np.sin(th), rng.uniform(-90, 300)], [s * np.sin(th), s * np.cos(th), rng.uniform(-40, 40)],
                              [0, 0, 1]], np.float32)
                cam, scale = rigs.Camera(1.0, 1.0, 0.0, 0.0, R), 1.0
            else:
                wide = wtype in ("spherical", "cylindrical")
                R = _rot(rng.uniform(-0.3, 0.3), rng.uniform(-3.0, 3.0) if wide else rng.uniform(-0.45, 0.45), rng.uniform(-0.15, 0.15))
                cam = rigs.Camera(rng.uniform(70, 120), rng.uniform(0.97, 1.03), W / 2 + rng.uniform(-4, 4), H / 2 + rng.uniform(-3, 3), R)
                scale = float(rng.uniform(60, 120))
            aspect = float(rng.choice([1.0, 0.8, 1.25])) if trial == 2 else 1.0
            img = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
            yield dict(key=f"proj_{wtype}_{trial}", wtype=wtype, trial=trial, cam=cam, scale=scale, aspect=aspect, img=img, size=(W, H))


def blend_cases(seed):
    rng = np.random.default_rng(seed)
    for trial in range(9):
        kind = ("multiband", "feather", "no")[trial % 3]
        strength = float(rng.choice([1, 5, 20, 60]))
        n = int(rng.integers(2, 5))
        sizes = [(int(rng.integers(40, 120)), int(rng.integers(30, 90))) for _ in range(n)]
        corners = [(int(rng.integers(-20, 20)) + 35 * i, int(rng.integers(-15, 15))) for i in range(n)]
        imgs = [rng.integers(0, 256, (h, w, 3), dtype=np.uint8) for (w, h) in sizes]
        masks = []
        for (w, h) in sizes:
            m = np.full((h, w), 255, np.uint8)
            if trial % 2:
                m[rng.random((h, w)) < 0.1] = 0
            if trial % 4 == 3:
                m = (m.astype(np.float32) * rng.random((h, w))).astype(np.uint8)  # gray seam-like masks
            masks.append(m)
        yield dict(key=f"blend_{trial}", kind=kind, strength=strength, sizes=sizes, corners=corners, imgs=imgs, masks=masks)


class _Scaler:
    def __init__(self, size):
        self.size = size

    def get_scaled_img_size(self, _):
        return self.size


def final_step_cases(seed, compensator_kinds):
    """SeamFinder.resize (seam_finder.py:38-43) and Images.resize_img_by_scaler (images.py:120-123) on random shapes;
    ExposureErrorCompensator.apply (exposure_error_compensator.py:43-45) of three overlapping exposures per compensator kind."""
    rng = np.random.default_rng(seed)
    for t in range(10):
        sh, sw = int(rng.integers(1, 70)), int(rng.integers(1, 90))
        h, w = int(rng.integers(2, 300)), int(rng.integers(2, 400))
        seam = (rng.integers(0, 256, (sh, sw), dtype=np.uint8) if t % 2 else (rng.random((sh, sw)) < 0.5).astype(np.uint8) * 255)
        mask = (rng.random((h, w)) < 0.85).astype(np.uint8) * 255
        yield dict(key=f"seam_{t}", step="seam_resize", seam=seam, mask=mask, what=f"SeamFinder.resize {sw}x{sh} -> {w}x{h}")
    for t in range(10):
        h, w = int(rng.integers(2, 200)), int(rng.integers(2, 260))
        size = (int(rng.integers(1, 300)), int(rng.integers(1, 240)))
        img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        yield dict(key=f"resize_{t}", step="img_resize", img=img, size=size, what=f"Images.resize {w}x{h} -> {size}")
    for kind in compensator_kinds:
        n = 3
        sizes = [(int(rng.integers(90, 160)), int(rng.integers(70, 120))) for _ in range(n)]
        corners = [(40 * i + int(rng.integers(-5, 5)), int(rng.integers(-5, 5))) for i in range(n)]
        base = rng.integers(30, 220, (200, 400, 3), dtype=np.uint8)
        imgs = []
        for i, ((w, h), (x, y)) in enumerate(zip(sizes, corners)):
            crop = base[20 + y: 20 + y + h, 20 + x: 20 + x + w].astype(np.float32) * (0.8 + 0.2 * i)
            imgs.append(np.clip(crop + rng.normal(0, 2, crop.shape), 0, 255).astype(np.uint8))
        masks = [np.full((h, w), 255, np.uint8) for (w, h) in sizes]
        yield dict(key=f"gain_{kind}", step="gain_apply", kind=kind, corners=corners, imgs=imgs, masks=masks)


DROPIN_RIGS = (("spherical", "multiband"), ("cylindrical", "feather"), ("plane", "no"), ("fisheye", "multiband"),
               ("paniniA2B1", "feather"), ("mercator", "multiband"), ("affine", "multiband"))


def dropin_cases(seed):
    rng = np.random.default_rng(seed)
    W, H = 120, 90
    for trial, (wtype, btype) in enumerate(DROPIN_RIGS):
        n = 3
        if wtype == "affine":
            cams = [rigs.Camera(1.0, 1.0, 0.0, 0.0, np.array([[1, 0.01 * i, 70.0 * i + rng.uniform(-3, 3)], [-0.01 * i, 1, rng.uniform(-8, 8)], [0, 0, 1]], np.float32))
                    for i in range(n)]
        else:
            f = rng.uniform(90, 130)
            cams = [rigs.Camera(f * rng.uniform(0.98, 1.02), 1.0, W / 2, H / 2, _rot(rng.uniform(-0.05, 0.05), 0.45 * (i - 1) + rng.uniform(-0.03, 0.03), rng.uniform(-0.03, 0.03)))
                    for i in range(n)]
        imgs = [rng.integers(0, 256, (H, W, 3), dtype=np.uint8) for _ in range(n)]
        yield dict(key=f"dropin_{trial}", wtype=wtype, btype=btype, cams=cams, imgs=imgs, sizes=[(W, H)] * n)


def run_dropin(case, Warper, Blender, Timelapser):
    """Warper (set_scale, warp_rois, warp_images, create_and_warp_masks) -> Blender (prepare, feed, blend) and a Timelapser frame
    of the same warped images, the calls stitcher.py makes."""
    cams, imgs = case["cams"], case["imgs"]
    w = Warper(case["wtype"])
    w.set_scale(cams)
    warped = list(w.warp_images(imgs, cams))
    masks = list(w.create_and_warp_masks(case["sizes"], cams))
    corners, wsizes = w.warp_rois(case["sizes"], cams)
    b = Blender(case["btype"], 5)
    b.prepare(corners, wsizes)
    for img, m, c in zip(warped, masks, corners):
        b.feed(img, m, c)
    pano, pmask = b.blend()
    t = Timelapser("as_is")
    t.initialize(corners, wsizes)
    t.process_frame(warped[1], corners[1])
    return dict(corners=np.array([[int(v) for v in c] for c in corners], np.int64), sizes=np.array([[int(v) for v in s] for s in wsizes], np.int64),
                warped=[np.asarray(x) for x in warped], masks=[np.asarray(x) for x in masks], pano=np.asarray(pano),
                pmask=np.asarray(pmask.get() if hasattr(pmask, "get") else pmask), frame=np.asarray(t.get_frame()))


def test_every_projection_against_the_reference_warper(oracle):
    g = replay.load(GOLDEN)
    types = [str(t) for t in g["warp_types"]]
    assert len(types) == 16
    checked = 0
    for c in projection_cases(int(g["seed"]), types):
        k, cam, scale, aspect, what = c["key"], c["cam"], c["scale"], c["aspect"], f"{c['wtype']} trial {c['trial']}"
        K = g[f"{k}_K"]  # Warper.get_K(camera, aspect) of the reference
        roi = tuple(int(v) for v in g[f"{k}_roi"])
        got_roi = oracle.warp_roi(c["wtype"], scale * aspect, K, cam.R, c["size"])
        assert tuple(got_roi) == roi, (what, got_roi, roi)
        if roi[2] * roi[3] > 4_000_000:
            continue  # a degenerate draw (horizon in view): the rect is exact, the pixels would take minutes
        rect, gimg, gmask = oracle.warp(c["wtype"], scale * aspect, K, cam.R, c["img"])
        replay.assert_golden(gimg, g, f"{k}_img", f"{what}: warped image")
        replay.assert_golden(gmask, g, f"{k}_mask", f"{what}: warped mask")
        checked += 1
    assert checked >= 40


def test_blenders_and_timelapser_against_the_reference(oracle):
    g = replay.load(GOLDEN)
    for c in blend_cases(int(g["seed"])):
        k, kind, strength, corners, sizes = c["key"], c["kind"], c["strength"], c["corners"], c["sizes"]
        b = oracle.Blender(kind, strength)
        b.prepare(corners, sizes)
        for img, m, corner in zip(c["imgs"], c["masks"], corners):
            b.feed(img, m, corner)
        pb, mb = b.blend()
        replay.assert_golden(np.asarray(pb), g, f"{k}_pano", f"{kind} strength {strength}: panorama")
        replay.assert_golden(np.asarray(mb), g, f"{k}_pmask", f"{kind} strength {strength}: mask")
        for tl_kind in ("as_is", "crop"):
            tb = oracle.Timelapser(tl_kind)
            tb.initialize(corners, sizes)
            for i, (img, corner) in enumerate(zip(c["imgs"], corners)):
                tb.process_frame(img, corner)
                key = f"{k}_{tl_kind}_{i}"
                if tb.roi[2] == 0 or tb.roi[3] == 0:  # rects that touch in a line: the reference's get_frame raises on the empty canvas
                    assert bool(g[f"{key}_raised"]), f"timelapse {tl_kind} frame {i}: empty canvas, but the reference returned a frame"
                    continue
                assert not bool(g[f"{key}_raised"]), f"timelapse {tl_kind} frame {i}: the reference raised"
                replay.assert_golden(tb.get_frame(), g, key, f"timelapse {tl_kind} frame {i}")


def test_final_resolution_steps_against_the_reference(oracle):
    """ExposureErrorCompensator.apply with the gains the reference's own feed() estimated."""
    g = replay.load(GOLDEN)
    kinds = [str(t) for t in g["compensator_kinds"]]
    for c in final_step_cases(int(g["seed"]), kinds):
        k = c["key"]
        if c["step"] == "seam_resize":
            replay.assert_golden(oracle.seam_resize(c["seam"], c["mask"]), g, k, c["what"])
        elif c["step"] == "img_resize":
            replay.assert_golden(oracle.resize_linear_exact(c["img"], c["size"]), g, k, c["what"])
        else:
            for i, img in enumerate(c["imgs"]):
                if c["kind"] == "no":
                    replay.assert_golden(img, g, f"{k}_{i}", "compensator no: identity")
                    continue
                replay.assert_golden(oracle.gain_apply(img, g[f"{k}_{i}_gain"]), g, f"{k}_{i}", f"compensator {c['kind']} image {i}")


def test_drop_in_classes_against_the_reference_classes(use_emu):
    """The product's own classes (their kernels through tests/emu) against what the reference's classes returned for the same
    calls and inputs: random rigs of every blender type and a handful of projections."""
    import stitching_b200

    g = replay.load(GOLDEN)
    for c in dropin_cases(int(g["seed"])):
        k, wtype, btype = c["key"], c["wtype"], c["btype"]
        b = run_dropin(c, stitching_b200.Warper, stitching_b200.Blender, stitching_b200.Timelapser)
        assert np.array_equal(b["corners"], g[f"{k}_corners"]) and np.array_equal(b["sizes"], g[f"{k}_sizes"]), \
            (wtype, b["corners"], g[f"{k}_corners"])
        for i in range(len(c["imgs"])):
            replay.assert_golden(b["warped"][i], g, f"{k}_warped_{i}", f"{wtype}: warped image {i}")
            replay.assert_golden(b["masks"][i], g, f"{k}_mask_{i}", f"{wtype}: warped mask {i}")
        replay.assert_golden(b["pano"], g, f"{k}_pano", f"{wtype} + {btype}: panorama")
        replay.assert_golden(b["pmask"], g, f"{k}_pmask", f"{wtype} + {btype}: panorama mask")
        replay.assert_golden(b["frame"], g, f"{k}_frame", f"{wtype}: timelapse frame")


def record(reference_dir, seed):
    """Run the reference classes on every case above and write what they returned to tests/golden/GOLDEN."""
    import cv2 as cv

    sys.path.insert(0, os.path.abspath(reference_dir))
    ref = importlib.import_module("stitching")
    for name in ("warper", "blender", "timelapser", "seam_finder", "images", "exposure_error_compensator"):
        importlib.import_module(f"stitching.{name}")
    types = list(ref.warper.Warper.WARP_TYPE_CHOICES)
    kinds = list(ref.exposure_error_compensator.ExposureErrorCompensator.COMPENSATOR_CHOICES)
    out = {"seed": np.int64(seed), "warp_types": np.array(types), "compensator_kinds": np.array(kinds), "cv2_version": cv.__version__}
    for c in projection_cases(seed, types):
        k = c["key"]
        wr = ref.warper.Warper(c["wtype"])
        wr.scale = c["scale"]
        out[f"{k}_K"] = ref.warper.Warper.get_K(c["cam"], c["aspect"])
        roi = tuple(int(v) for v in wr.warp_roi(c["size"], c["cam"], c["aspect"]))
        out[f"{k}_roi"] = np.array(roi, np.int64)
        if roi[2] * roi[3] > 4_000_000:
            continue
        replay.pack(out, f"{k}_img", wr.warp_image(c["img"], c["cam"], c["aspect"]))
        replay.pack(out, f"{k}_mask", wr.create_and_warp_mask(c["size"], c["cam"], c["aspect"]))
    for c in blend_cases(seed):
        k = c["key"]
        a = ref.blender.Blender(c["kind"], c["strength"])
        a.prepare(c["corners"], c["sizes"])
        for img, m, corner in zip(c["imgs"], c["masks"], c["corners"]):
            a.feed(img, m, corner)
        pa, ma = a.blend()
        replay.pack(out, f"{k}_pano", np.asarray(pa))
        replay.pack(out, f"{k}_pmask", np.asarray(ma.get() if hasattr(ma, "get") else ma))
        for tl_kind in ("as_is", "crop"):
            ta = ref.timelapser.Timelapser(tl_kind)
            ta.initialize(c["corners"], c["sizes"])
            for i, (img, corner) in enumerate(zip(c["imgs"], c["corners"])):
                ta.process_frame(img, corner)
                key = f"{k}_{tl_kind}_{i}"
                try:
                    replay.pack(out, key, ta.get_frame())
                    out[f"{key}_raised"] = np.bool_(False)
                except cv.error:
                    out[f"{key}_raised"] = np.bool_(True)
    for c in final_step_cases(seed, kinds):
        k = c["key"]
        if c["step"] == "seam_resize":
            want = ref.seam_finder.SeamFinder.resize(cv.UMat(c["seam"]), c["mask"])
            replay.pack(out, k, want.get() if hasattr(want, "get") else np.asarray(want))
        elif c["step"] == "img_resize":
            w, h = c["img"].shape[1], c["img"].shape[0]
            replay.pack(out, k, ref.images.Images.resize_img_by_scaler(_Scaler(c["size"]), (w, h), c["img"]))
        else:
            comp = ref.exposure_error_compensator.ExposureErrorCompensator(c["kind"], 1, 16)
            comp.feed(c["corners"], c["imgs"], c["masks"])
            for i, img in enumerate(c["imgs"]):
                if c["kind"] != "no":
                    out[f"{k}_{i}_gain"] = np.asarray(comp.compensator.getMatGains()[i])
                replay.pack(out, f"{k}_{i}", comp.apply(i, c["corners"][i], img.copy(), c["masks"][i]))
    for c in dropin_cases(seed):
        k = c["key"]
        a = run_dropin(c, ref.warper.Warper, ref.blender.Blender, ref.timelapser.Timelapser)
        out[f"{k}_corners"], out[f"{k}_sizes"] = a["corners"], a["sizes"]
        for i in range(len(c["imgs"])):
            replay.pack(out, f"{k}_warped_{i}", a["warped"][i])
            replay.pack(out, f"{k}_mask_{i}", a["masks"][i])
        for name in ("pano", "pmask", "frame"):
            replay.pack(out, f"{k}_{name}", a[name])
    np.savez_compressed(os.path.join(replay.GOLDEN, GOLDEN), **out)


if __name__ == "__main__":
    record(sys.argv[1], int(sys.argv[2]) if len(sys.argv) > 2 else 20260923)
