"""Drop-in check against the real reference pipeline.

stitching.Stitcher(crop=False) runs unmodified on three synthetic perspective views of a textured plane.  The
reference's registration is not deterministic from run to run (RANSAC), so two whole runs cannot be compared;
instead every call that crosses the hot-path boundary (Warper, SeamFinder.resize, Blender) was RECORDED while the reference ran with its
own classes (the cameras, aspects, blend masks and corners it hands over, with the container type of every image argument, and
what cv2 returned; stored in tests/golden/golden_dropin.npz, written by write_golden), and is REPLAYED through the B200 classes
(here on the emulation build, tests/emu) with arguments of the same types: cv.detail.CameraParams rebuilt from the recorded
focal, aspect, principal point and R, numpy-float aspects, cv.UMat where the pipeline passed cv.UMat.  Every warped image,
mask, roi and the final panorama must be identical.  A second part
runs the whole pipeline with stitching_b200.install() to show that it executes end to end on the swapped classes; it needs
the reference package (OpenStitching/stitching): oracle/_ref, which build() compiles from a reference checkout, or an
installed `stitching`.
"""
import hashlib
import importlib
import os
import sys

import numpy as np
import pytest

import replay

GOLDEN = "golden_dropin.npz"


@pytest.fixture()
def reference_stitching():
    """The reference package, fresh for every test (install() patches it): from oracle/_ref, which build() compiles from a
    reference checkout (oracle/reference.py), or else an installed `stitching`."""
    from oracle import reference

    cv = pytest.importorskip("cv2")
    ref_dir = reference.REF_DIR if os.path.isfile(os.path.join(reference.REF_DIR, "stitching", "__init__.pyc")) else None
    if ref_dir:
        sys.path.insert(0, ref_dir)
    for name in [m for m in sys.modules if m == "stitching" or m.startswith("stitching.")]:
        del sys.modules[name]
    try:
        if ref_dir:  # built here: it has to import (a .pyc of another Python version fails here instead of skipping)
            yield importlib.import_module("stitching"), cv
        else:
            yield pytest.importorskip("stitching", reason="no reference package: neither oracle/_ref (build() with a reference "
                                                          "checkout) nor an installed one"), cv
    finally:
        for name in [m for m in sys.modules if m == "stitching" or m.startswith("stitching.")]:
            del sys.modules[name]
        if ref_dir:
            sys.path.remove(ref_dir)


def synthetic_views(cv):
    rng = np.random.default_rng(5)
    scene = np.zeros((1400, 3000, 3), np.uint8)
    scene[:] = cv.resize(rng.integers(0, 256, (24, 50, 3), dtype=np.uint8), (3000, 1400), interpolation=cv.INTER_CUBIC)
    for _ in range(900):  # random shapes give ORB something to hold on to
        c = tuple(int(v) for v in rng.integers(0, 256, 3))
        p = (int(rng.integers(0, 3000)), int(rng.integers(0, 1400)))
        if rng.random() < 0.5:
            cv.circle(scene, p, int(rng.integers(5, 40)), c, -1)
        else:
            q = (p[0] + int(rng.integers(10, 90)), p[1] + int(rng.integers(10, 90)))
            cv.rectangle(scene, p, q, c, -1)
    views = []
    f, w, h = 900.0, 1000, 750
    K = np.array([[f, 0, w / 2], [0, f, h / 2], [0, 0, 1]])
    Ks = np.array([[f, 0, 1500], [0, f, 700], [0, 0, 1]])
    for yaw in (-0.35, 0.0, 0.35):
        R = np.array([[np.cos(yaw), 0, np.sin(yaw)], [0, 1, 0], [-np.sin(yaw), 0, np.cos(yaw)]])
        H = K @ R @ np.linalg.inv(Ks)
        views.append(cv.warpPerspective(scene, H, (w, h)))
    # different exposures, so that the exposure compensator has something to do
    views[0] = np.clip(views[0].astype(np.float32) * 0.82, 0, 255).astype(np.uint8)
    views[2] = np.clip(views[2].astype(np.float32) * 1.12, 0, 255).astype(np.uint8)
    return views


SETTINGS = dict(crop=False, detector="orb", confidence_threshold=0.3)


def record_boundary_calls(stitching, cv):
    """Run stitching.Stitcher with its own classes and log every call that crosses the hot-path boundary."""
    from stitching.blender import Blender as RefBlender
    from stitching.warper import Warper as RefWarper

    log = []

    class RecWarper(RefWarper):
        def warp_image(self, img, camera, aspect=1):
            out = super().warp_image(img, camera, aspect)
            log.append(("warp_image", self.warper_type, self.scale, np.array(img).copy(), camera, aspect, out.copy()))
            return out

        def create_and_warp_mask(self, size, camera, aspect=1):
            out = super().create_and_warp_mask(size, camera, aspect)
            log.append(("warp_mask", self.warper_type, self.scale, tuple(size), camera, aspect, out.copy()))
            return out

        def warp_roi(self, size, camera, aspect=1):
            out = super().warp_roi(size, camera, aspect)
            log.append(("warp_roi", self.warper_type, self.scale, tuple(size), camera, aspect, tuple(out)))
            return out

    class RecBlender(RefBlender):
        def prepare(self, corners, sizes):
            log.append(("prepare", self.blender_type, self.blend_strength, list(corners), list(sizes)))
            super().prepare(corners, sizes)

        def feed(self, img, mask, corner):
            log.append(("feed", np.array(img).copy(), mask, tuple(corner)))  # mask stays the cv.UMat the pipeline passes
            super().feed(img, mask, corner)

        def blend(self):
            pano, mask = super().blend()
            log.append(("blend", pano.copy(), np.array(mask).copy()))
            return pano, mask

    from stitching.seam_finder import SeamFinder as RefSeamFinder

    ref_resize = RefSeamFinder.resize

    def rec_resize(seam_mask, mask):
        out = ref_resize(seam_mask, mask)
        log.append(("seam_resize", seam_mask, np.array(mask).copy(), out.get() if hasattr(out, "get") else np.array(out), type(out).__name__))
        return out

    from stitching.exposure_error_compensator import ExposureErrorCompensator as RefCompensator

    ref_apply = RefCompensator.apply

    def rec_apply(self, *args):
        idx, _corner, img, _mask = args
        before = np.array(img).copy()
        gain = np.array(self.compensator.getMatGains()[idx]).copy()
        out = ref_apply(self, *args)
        log.append(("gain_apply", gain, before, np.array(out.get() if hasattr(out, "get") else out).copy()))
        return out

    from stitching.images import Images as RefImages

    ref_img_resize = RefImages.resize_img_by_scaler

    def rec_img_resize(scaler, size, img):
        out = ref_img_resize(scaler, size, img)
        log.append(("img_resize", np.array(img).copy(), scaler.get_scaled_img_size(size), np.array(out).copy()))
        return out

    stitching.stitcher.Warper, stitching.stitcher.Blender = RecWarper, RecBlender
    RefSeamFinder.resize = staticmethod(rec_resize)
    RefCompensator.apply = rec_apply
    RefImages.resize_img_by_scaler = staticmethod(rec_img_resize)
    try:
        stitching.Stitcher(**SETTINGS).stitch([v.copy() for v in synthetic_views(cv)])
    finally:
        RefSeamFinder.resize = staticmethod(ref_resize)
        RefCompensator.apply = ref_apply
        RefImages.resize_img_by_scaler = staticmethod(ref_img_resize)
    kinds = [e[0] for e in log]
    assert kinds.count("warp_image") >= 6 and kinds.count("feed") == 3 and kinds.count("blend") == 1
    assert kinds.count("seam_resize") == 3, "stitcher.py:223-225 resizes one seam mask per image"
    assert kinds.count("img_resize") >= 6, "images.py:120-123 resamples every image to the working resolutions"
    applied = [e for e in log if e[0] == "gain_apply"]
    assert len(applied) == 3 and any(not np.array_equal(e[2], e[3]) for e in applied), "stitcher.py:219-221 compensates every image"
    assert any(type(e[2]).__name__ == "UMat" for e in log if e[0] == "feed"), "the pipeline hands cv.UMat masks to feed"
    return log


def _sha(arr):
    return hashlib.sha256(np.ascontiguousarray(arr).tobytes()).hexdigest()


def write_golden(stitching, cv):
    """Store one recorded run in tests/golden/GOLDEN: per call its arguments and what the reference returned (replay.pack).
    An image argument that the synthetic views or an earlier call's result already is, is stored as that name
    ("view_<i>", "out_<k>"); the others (the LOW-resolution seam masks of the graph cut, the gains) are stored whole."""
    views = synthetic_views(cv)
    log = record_boundary_calls(stitching, cv)
    known = {_sha(v): f"view_{i}" for i, v in enumerate(views)}
    out = {"n": np.int64(len(log)), "views_sha256": np.array([_sha(v) for v in views])}

    def arg(k, name, arr):
        out[f"e{k}_{name}_type"] = "UMat" if isinstance(arr, cv.UMat) else "ndarray"
        arr = np.asarray(arr.get() if isinstance(arr, cv.UMat) else arr)
        src = known.get(_sha(arr))
        if src is None:
            out[f"e{k}_{name}"] = arr
        else:
            out[f"e{k}_{name}_from"] = src

    def result(k, arr):
        replay.pack(out, f"e{k}_out", arr)
        known.setdefault(_sha(arr), f"out_{k}")

    for k, e in enumerate(log):
        out[f"e{k}_kind"] = e[0]
        if e[0] in ("warp_image", "warp_mask", "warp_roi"):
            cam = e[4]
            out[f"e{k}_warper"], out[f"e{k}_scale"], out[f"e{k}_aspect"] = e[1], np.float64(e[2]), np.float64(e[5])
            out[f"e{k}_camera"] = np.array([cam.focal, cam.aspect, cam.ppx, cam.ppy], np.float64)
            out[f"e{k}_R"] = np.asarray(cam.R)
            if e[0] == "warp_image":
                arg(k, "img", e[3])
                result(k, e[6])
            else:
                out[f"e{k}_size"] = np.array(e[3], np.int64)
                if e[0] == "warp_mask":
                    result(k, e[6])
                else:
                    out[f"e{k}_out"] = np.array(e[6], np.int64)
        elif e[0] == "img_resize":
            arg(k, "img", e[1])
            out[f"e{k}_size"] = np.array(e[2], np.int64)
            result(k, e[3])
        elif e[0] == "gain_apply":
            out[f"e{k}_gain"] = e[1]
            arg(k, "img", e[2])
            result(k, e[3])
        elif e[0] == "seam_resize":
            arg(k, "seam", e[1])
            arg(k, "mask", e[2])
            out[f"e{k}_out_type"] = e[4]
            result(k, e[3])
        elif e[0] == "prepare":
            out[f"e{k}_blender"], out[f"e{k}_strength"] = e[1], np.float64(e[2])
            out[f"e{k}_corners"], out[f"e{k}_sizes"] = np.array(e[3], np.int64), np.array(e[4], np.int64)
        elif e[0] == "feed":
            arg(k, "img", e[1])
            arg(k, "mask", e[2])
            out[f"e{k}_corner"] = np.array(e[3], np.int64)
        elif e[0] == "blend":
            replay.pack(out, f"e{k}_out", e[1])
            replay.pack(out, f"e{k}_mask", e[2])
    np.savez_compressed(os.path.join(replay.GOLDEN, GOLDEN), **out)


def test_recorded_boundary_calls_replay_identically(use_emu):
    """The calls one reference run made (GOLDEN, written by write_golden) replayed through the B200 classes."""
    cv = pytest.importorskip("cv2")
    import stitching_b200

    g = replay.load(GOLDEN)
    views = synthetic_views(cv)
    assert [_sha(v) for v in views] == [str(s) for s in g["views_sha256"]], "synthetic_views drifted from the recorded run"
    results = {f"view_{i}": v for i, v in enumerate(views)}

    def arg(k, name):
        arr = results[str(g[f"e{k}_{name}_from"])] if f"e{k}_{name}_from" in g.files else g[f"e{k}_{name}"]
        return cv.UMat(arr) if str(g[f"e{k}_{name}_type"]) == "UMat" else arr

    def camera(k):
        cam = cv.detail.CameraParams()
        cam.focal, cam.aspect, cam.ppx, cam.ppy = (float(v) for v in g[f"e{k}_camera"])
        cam.R = g[f"e{k}_R"]
        return cam

    kinds = [str(g[f"e{k}_kind"]) for k in range(int(g["n"]))]
    assert kinds.count("warp_image") >= 6 and kinds.count("feed") == 3 and kinds.count("blend") == 1
    assert kinds.count("seam_resize") == 3 and kinds.count("img_resize") >= 6 and kinds.count("gain_apply") == 3
    assert any(str(g[f"e{k}_mask_type"]) == "UMat" for k, kind in enumerate(kinds) if kind == "feed"), "the pipeline hands cv.UMat masks to feed"
    blender = None
    checked = compensated = 0
    for k, kind in enumerate(kinds):
        what = f"call {k} ({kind})"
        if kind in ("warp_image", "warp_mask", "warp_roi"):
            w = stitching_b200.Warper(str(g[f"e{k}_warper"]))
            w.scale = float(g[f"e{k}_scale"])
            cam, aspect = camera(k), np.float64(g[f"e{k}_aspect"])  # the numpy float the pipeline hands over
            if kind == "warp_roi":
                assert tuple(w.warp_roi(tuple(int(v) for v in g[f"e{k}_size"]), cam, aspect)) == tuple(int(v) for v in g[f"e{k}_out"]), what
            else:
                got = w.warp_image(arg(k, "img"), cam, aspect) if kind == "warp_image" else \
                    w.create_and_warp_mask(tuple(int(v) for v in g[f"e{k}_size"]), cam, aspect)
                replay.assert_golden(got, g, f"e{k}_out", what)
                results[f"out_{k}"] = got
            checked += 1
        elif kind == "img_resize":  # images.py:120-123: the MEDIUM / LOW / FINAL resolution inputs
            got = stitching_b200.images.resize_exact(arg(k, "img"), tuple(int(v) for v in g[f"e{k}_size"]))
            replay.assert_golden(got, g, f"e{k}_out", f"{what}: Images.resize")
            results[f"out_{k}"] = got
            checked += 1
        elif kind == "gain_apply":  # the default compensator (gain_blocks) with the gains its own feed() estimated
            before = arg(k, "img")
            got = stitching_b200.exposure_error_compensator.apply_gain(before.copy(), g[f"e{k}_gain"])
            replay.assert_golden(got, g, f"e{k}_out", f"{what}: ExposureErrorCompensator.apply")
            compensated += not np.array_equal(got, before)
            results[f"out_{k}"] = got
            checked += 1
        elif kind == "seam_resize":  # the LOW-resolution seam mask arrives as cv.UMat, the warped mask as ndarray
            got = stitching_b200.seam_finder.resize(arg(k, "seam"), arg(k, "mask"))
            # same container type as the reference's cv2 chain (cv.UMat in the pipeline): seam_finder.py:47 and
            # verbose.py:149-156 call cv.UMat.get on it
            assert type(got).__name__ == str(g[f"e{k}_out_type"]), f"SeamFinder.resize returned {type(got).__name__}, the reference {g[f'e{k}_out_type']}"
            got = got.get() if hasattr(got, "get") else got
            replay.assert_golden(got, g, f"e{k}_out", f"{what}: SeamFinder.resize")
            results[f"out_{k}"] = got
            checked += 1
        elif kind == "prepare":
            blender = stitching_b200.Blender(str(g[f"e{k}_blender"]), float(g[f"e{k}_strength"]))
            blender.prepare([tuple(int(v) for v in c) for c in g[f"e{k}_corners"]], [tuple(int(v) for v in s) for s in g[f"e{k}_sizes"]])
        elif kind == "feed":
            blender.feed(arg(k, "img"), arg(k, "mask"), tuple(int(v) for v in g[f"e{k}_corner"]))
        elif kind == "blend":
            pano, mask = blender.blend()
            replay.assert_golden(mask, g, f"e{k}_mask", "panorama mask")
            replay.assert_golden(pano, g, f"e{k}_out", "panorama")
            checked += 1
    assert compensated > 0, "stitcher.py:219-221 compensates every image"
    assert checked >= 19


def test_stitcher_runs_end_to_end_on_the_swapped_classes(reference_stitching, use_emu):
    stitching, cv = reference_stitching
    import stitching_b200

    views = synthetic_views(cv)
    ref_pano = stitching.Stitcher(**SETTINGS).stitch([v.copy() for v in views])
    stitching_b200.install(stitching)
    assert stitching.stitcher.Warper is stitching_b200.Warper and stitching.stitcher.Blender is stitching_b200.Blender
    # the package surface of stitching/__init__.py:1, with the reference's own settings
    assert stitching_b200.Stitcher is stitching.Stitcher and stitching_b200.AffineStitcher is stitching.AffineStitcher
    assert stitching_b200.Stitcher.DEFAULT_SETTINGS["warper_type"] == "spherical"
    pano = stitching.Stitcher(**SETTINGS).stitch([v.copy() for v in views])
    # registration is re-estimated (RANSAC): same geometry up to a few pixels, same kind of picture
    assert pano.ndim == 3 and pano.dtype == np.uint8
    assert abs(pano.shape[0] - ref_pano.shape[0]) <= 30 and abs(pano.shape[1] - ref_pano.shape[1]) <= 30  # tests/test_stitcher.py:229-231 style
    assert (pano.sum(axis=2) > 0).mean() > 0.5


def test_stitch_verbose_runs_after_install(reference_stitching, use_emu, tmp_path):
    """Stitcher.stitch_verbose (verbose.py) after install(): it draws the FINAL-resolution seam masks with
    SeamFinder.draw_seam_mask, i.e. cv.UMat.get(seam_mask) (seam_finder.py:47, verbose.py:149-156) -- the drop-in
    SeamFinder.resize therefore has to hand out what the reference hands out (a cv.UMat)."""
    stitching, cv = reference_stitching
    import stitching_b200

    stitching_b200.install(stitching)
    views = synthetic_views(cv)
    pano = stitching.Stitcher(**SETTINGS).stitch_verbose([v.copy() for v in views], verbose_dir=str(tmp_path))
    assert pano.ndim == 3 and pano.dtype == np.uint8 and (pano.sum(axis=2) > 0).mean() > 0.5
    written = sorted(os.listdir(tmp_path))
    assert any(name.startswith("08_seam_mask") for name in written) and "09_result.jpg" in written, written


@pytest.mark.parametrize("warper_type", ["fisheye", "compressedPlaneA2B1"])  # the two the reference's own tests use (tests/test_stitcher.py:85,110)
def test_stitcher_with_other_warper_types_after_install(reference_stitching, use_emu, warper_type):
    stitching, cv = reference_stitching
    import stitching_b200

    views = synthetic_views(cv)
    ref_pano = stitching.Stitcher(warper_type=warper_type, **SETTINGS).stitch([v.copy() for v in views])
    stitching_b200.install(stitching)
    pano = stitching.Stitcher(warper_type=warper_type, **SETTINGS).stitch([v.copy() for v in views])
    assert pano.ndim == 3 and pano.dtype == np.uint8 and (pano.sum(axis=2) > 0).mean() > 0.3
    assert abs(pano.shape[0] - ref_pano.shape[0]) <= 40 and abs(pano.shape[1] - ref_pano.shape[1]) <= 40


def test_timelapse_run_after_install(reference_stitching, use_emu, tmp_path):
    """Stitcher(timelapse="as_is") after install(): the warped FINAL-resolution frames go to the drop-in Timelapser
    (stitcher.py:242-252) instead of the blender; one "fixed_" file per input appears next to the inputs, each the frame of
    the whole panorama roi with one image in it."""
    stitching, cv = reference_stitching
    import stitching_b200

    views = synthetic_views(cv)
    names = []
    for i, v in enumerate(views):
        names.append(str(tmp_path / f"view{i}.png"))
        cv.imwrite(names[-1], v)
    stitching_b200.install(stitching)
    assert stitching.stitcher.Timelapser is stitching_b200.Timelapser
    out = stitching.Stitcher(timelapse="as_is", **SETTINGS).stitch(names)
    assert out is None  # create_final_panorama returns nothing in timelapse mode (stitcher.py:257-260)
    frames = [cv.imread(str(tmp_path / f"fixed_view{i}.png")) for i in range(len(views))]
    assert all(f is not None and f.shape == frames[0].shape for f in frames)
    cover = [(f.sum(axis=2) > 0) for f in frames]
    assert all(0.1 < c.mean() < 0.9 for c in cover)                     # one image per frame, not the panorama
    centres = [np.nonzero(c.any(axis=0))[0].mean() for c in cover]
    assert min(abs(a - b) for i, a in enumerate(centres) for b in centres[i + 1:]) > 100  # three different places on the canvas


def test_one_stitcher_for_two_image_sets_and_affine_stitcher_after_install(reference_stitching, use_emu):
    """tests/test_stitcher.py:283-290 re-uses one Stitcher for two image sets, :173-185 runs AffineStitcher (plane warp
    through the affine warper, feather-free defaults): both after install(), on the swapped classes."""
    stitching, cv = reference_stitching
    import stitching_b200

    stitching_b200.install(stitching)
    views = synthetic_views(cv)
    st = stitching.Stitcher(**SETTINGS)
    first = st.stitch([v.copy() for v in views])
    second = st.stitch([v.copy() for v in views[:2]])            # a different set through the same object
    assert first.ndim == 3 and second.ndim == 3 and second.shape[1] < first.shape[1]
    again = st.stitch([v.copy() for v in views])
    assert abs(again.shape[0] - first.shape[0]) <= 30 and abs(again.shape[1] - first.shape[1]) <= 30

    # AffineStitcher: flat scans of one scene, shifted and slightly rotated against each other
    rng = np.random.default_rng(11)
    scene = cv.resize(rng.integers(0, 256, (30, 40, 3), dtype=np.uint8), (1600, 1200), interpolation=cv.INTER_CUBIC)
    for _ in range(700):
        c = tuple(int(v) for v in rng.integers(0, 256, 3))
        p = (int(rng.integers(0, 1600)), int(rng.integers(0, 1200)))
        cv.circle(scene, p, int(rng.integers(4, 30)), c, -1)
    scans = []
    for dx, ang in ((0, 0.0), (380, 1.5), (760, -1.0)):
        M = cv.getRotationMatrix2D((400, 500), ang, 1.0)
        M[0, 2] -= dx
        scans.append(cv.warpAffine(scene, M, (800, 1000)))
    try:
        pano = stitching.AffineStitcher(crop=False, detector="orb", confidence_threshold=0.3).stitch(scans)
    except stitching.stitching_error.StitchingError as e:  # registration is the reference's business; tell, do not fail
        pytest.skip(f"the reference could not register the synthetic scans: {e}")
    assert pano.ndim == 3 and pano.dtype == np.uint8
    assert pano.shape[1] > 1200 and (pano.sum(axis=2) > 0).mean() > 0.5  # wider than one scan: the scans were composed


if __name__ == "__main__":  # PYTHONPATH=.:tests:<reference checkout> python tests/test_dropin_pipeline.py
    import cv2

    import stitching

    write_golden(stitching, cv2)
