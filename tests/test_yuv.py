"""YUV 4:2:0 frames (NV12 / I420) in and out of the compositor, on a GPU-less box.

The contract (DESIGN.md section 2): a YUV input frame means cv.cvtColor(frame, COLOR_YUV2BGR_NV12 / _I420) followed by
the BGR pipeline; a YUV panorama means cv.cvtColor(pano, COLOR_BGR2YUV_I420) of the BGR panorama, U and V interleaved
for NV12.  tests/yuv_oracle.py restates both conversions; it is checked against cv2 live (when installed) and against
tests/golden/golden_yuv.npz, and the product's kernels (sb_yuv.cu, through tests/emu) against it.  The check_* functions
take the library in use and are shared with tests/test_gpu_yuv.py, which runs them on the B200.
"""
import ctypes as C
import os

import numpy as np
import pytest

import yuv_oracle as YO
from stitching_b200 import Compositor, StitchingError, _lib, color, rigs

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "golden_yuv.npz")
FMTS = ("bgr", "nv12", "i420")
SB_ERR_INVALID, SB_ERR_STATE = -1, -4


def random_frame(w, h, fmt, seed):
    rng = np.random.default_rng(seed)
    if fmt == "bgr":
        return rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    return rng.integers(0, 256, (h * 3 // 2, w), dtype=np.uint8)


def to_bgr(frame, fmt):
    return frame if fmt == "bgr" else YO.yuv420_to_bgr(frame, fmt)


def from_bgr(img, fmt):
    return img if fmt == "bgr" else YO.bgr_to_yuv420(img, fmt)


def small_rig(name="cfg2", scale_down=20, n=None, warper=None):
    cfg = rigs.config(name, scale_down)
    cams = cfg["cameras"][:n] if n else cfg["cameras"]
    sizes = [(cfg["w"], cfg["h"])] * len(cams)
    return cfg, cams, sizes, (warper or cfg["warper"])


# ---- checks shared with tests/test_gpu_yuv.py ------------------------------------------------------------------------
def check_golden_through_library():
    z = np.load(GOLDEN)
    names = sorted({k.split("__")[0] for k in z.files})
    for name in names:
        kind, x, want = name.split("_")[0], z[name + "__in"], z[name + "__out"]
        if kind == "bgr":
            for fmt in ("i420", "nv12"):
                got = color.bgr_to_yuv420(x, fmt)
                exp = want if fmt == "i420" else YO.join(*YO.split(want, "i420"), "nv12")
                assert np.array_equal(got, exp), f"{name} -> {fmt}"
        else:
            assert np.array_equal(color.yuv420_to_bgr(x, kind), want), name


def check_exhaustive_frame_through_library():
    for fmt in ("nv12", "i420"):
        frame = YO.exhaustive_frame(fmt)
        exp = YO.yuv420_to_bgr(frame, fmt)
        got = color.yuv420_to_bgr(frame, fmt)
        assert np.array_equal(got, exp), f"{fmt}: {int((got != exp).sum())} values differ"
        back = color.bgr_to_yuv420(exp, fmt)
        assert np.array_equal(back, YO.bgr_to_yuv420(exp, fmt)), f"{fmt} BGR -> YUV of the exhaustive frame's colours"


def check_random_conversions_through_library():
    for k, (w, h) in enumerate(((2, 2), (6, 4), (130, 66), (642, 480))):
        img = random_frame(w, h, "bgr", k)
        img[: h // 2, : w // 2] = 255 * (img[: h // 2, : w // 2] > 127)  # saturated corners of the colour cube
        for fmt in ("nv12", "i420"):
            assert np.array_equal(color.bgr_to_yuv420(img, fmt), YO.bgr_to_yuv420(img, fmt)), f"{w}x{h} BGR -> {fmt}"
            frame = random_frame(w, h, fmt, 100 + k)
            assert np.array_equal(color.yuv420_to_bgr(frame, fmt), YO.yuv420_to_bgr(frame, fmt)), f"{w}x{h} {fmt} -> BGR"
    # strided views: rows of a wider buffer
    big = random_frame(64, 40, "bgr", 9)
    view = big[:, :32]
    assert np.array_equal(color.bgr_to_yuv420(view, "nv12"), YO.bgr_to_yuv420(view, "nv12"))
    nv = random_frame(64, 40, "nv12", 10)[:, :32]
    assert np.array_equal(color.yuv420_to_bgr(nv, "nv12"), YO.yuv420_to_bgr(nv, "nv12"))


def check_upload_equals_oracle_bgr_upload(monkeypatch, name="cfg2", scale_down=20, n=4, warper=None):
    """upload(fmt=YUV) + run == upload(oracle BGR of the same frames) + run, for both source layouts of the warp kernel."""
    cfg, cams, sizes, warper = small_rig(name, scale_down, n, warper)
    for flag in ("1", "0"):
        monkeypatch.setenv("SB_SRC4", flag)
        c = Compositor(cams, sizes, warper, cfg["blender"], cfg["strength"])
        for fmt in ("nv12", "i420"):
            frames = [random_frame(cfg["w"], cfg["h"], fmt, 50 + i) for i in range(len(cams))]
            exp_pano, exp_mask = (a.copy() for a in c.composite([YO.yuv420_to_bgr(f, fmt) for f in frames]))
            c.upload(frames, fmt=fmt)
            c.run()
            pano, mask = c.download()
            assert np.array_equal(pano, exp_pano) and np.array_equal(mask, exp_mask), f"{name} {warper} {fmt} SB_SRC4={flag}"
            wi, _ = c.download_warped(len(cams) - 1)
            c.upload([YO.yuv420_to_bgr(f, fmt) for f in frames])
            c.run()
            assert np.array_equal(wi, c.download_warped(len(cams) - 1)[0])
        c.close()


def check_download_equals_oracle(name="cfg2", scale_down=20, n=None):
    cfg, cams, sizes, warper = small_rig(name, scale_down, n)
    c = Compositor(cams, sizes, warper, cfg["blender"], cfg["strength"])
    imgs = [rigs.noise_image(cfg["h"], cfg["w"], 60 + i) for i in range(len(cams))]
    pano, mask = (a.copy() for a in c.composite(imgs))
    for fmt in ("nv12", "i420"):
        got, gmask = c.download(fmt=fmt)
        assert np.array_equal(got, YO.bgr_to_yuv420(pano, fmt)), fmt
        assert np.array_equal(gmask, mask)
        # a caller's output array, and the composite() shortcut
        out = np.empty_like(got)
        assert c.download(out=out, fmt=fmt)[0] is out and np.array_equal(out, got)
        p2, m2 = c.composite(imgs, out_fmt=fmt)
        assert np.array_equal(p2, got) and np.array_equal(m2, mask)
    c.close()


def check_submit_all_format_pairs(name="cfg2", scale_down=20, n=None, steps=2):
    """submit over all nine (in, out) format pairs, pipelined, equals composite of the same frames."""
    cfg, cams, sizes, warper = small_rig(name, scale_down, n)
    c = Compositor(cams, sizes, warper, cfg["blender"], cfg["strength"])
    _, _, pw, ph = c.roi
    jobs = [(fi, fo, s) for fi in FMTS for fo in FMTS for s in range(steps)]
    expected, inputs = [], []
    for k, (fi, fo, s) in enumerate(jobs):
        frames = [random_frame(cfg["w"], cfg["h"], fi, 1000 * k + i) for i in range(len(cams))]
        inputs.append(frames)
        expected.append(tuple(a.copy() for a in c.composite(frames, in_fmt=fi, out_fmt=fo)))
        if s == 0:  # the definition, once per pair: BGR composite of the oracle-converted frames, oracle-converted back
            bp, bm = c.composite([to_bgr(f, fi) for f in frames])
            assert np.array_equal(expected[-1][0], from_bgr(bp, fo)) and np.array_equal(expected[-1][1], bm), (fi, fo)
    depth = 3
    outs = {}
    tickets = []
    for k, (fi, fo, s) in enumerate(jobs):
        if k >= depth:
            done = k - depth
            c.wait(tickets[done])
            o = outs.pop(done)
            assert np.array_equal(o[0], expected[done][0]) and np.array_equal(o[1], expected[done][1]), jobs[done]
        o = (np.empty(color.frame_shape(pw, ph, fo), np.uint8), np.empty((ph, pw), np.uint8))
        outs[k] = o
        tickets.append(c.submit(inputs[k], o[0], o[1], in_fmt=fi, out_fmt=fo))
    for k in range(len(jobs) - depth, len(jobs)):
        c.wait(tickets[k])
        assert np.array_equal(outs[k][0], expected[k][0]) and np.array_equal(outs[k][1], expected[k][1]), jobs[k]
    # no mask, and no panorama
    fr = inputs[-1]
    o = np.empty(color.frame_shape(pw, ph, "nv12"), np.uint8)
    c.wait(c.submit(inputs[jobs.index(("i420", "nv12", 0))], o, None, in_fmt="i420", out_fmt="nv12"))
    assert np.array_equal(o, expected[jobs.index(("i420", "nv12", 0))][0])
    m = np.empty((ph, pw), np.uint8)
    c.wait(c.submit(fr, None, m, in_fmt="i420", out_fmt="nv12"))
    assert np.array_equal(m, expected[-1][1])
    c.close()


def check_error_cases():
    L = _lib.lib()
    u8 = np.zeros(16, np.uint8)

    def planes(ptr=u8.ctypes.data, pitch=64):
        return (C.c_void_p * 3)(ptr, ptr, ptr), (C.c_size_t * 3)(pitch, pitch, pitch)

    # the direct conversions: odd sizes, short pitches, missing planes, unknown formats
    p, q = planes()
    dst = np.zeros((8, 8, 3), np.uint8)
    for fmt in (1, 2):
        for w, h in ((5, 4), (4, 5), (0, 4)):
            assert L.sb_cvt_yuv420_to_bgr(fmt, p, q, w, h, dst.ctypes.data, 64) == SB_ERR_INVALID
            assert b"even" in L.sb_last_error()
            assert L.sb_cvt_bgr_to_yuv420(fmt, dst.ctypes.data, 64, w, h, p, q) == SB_ERR_INVALID
        _, short = planes(pitch=2)
        assert L.sb_cvt_yuv420_to_bgr(fmt, p, short, 8, 4, dst.ctypes.data, 64) == SB_ERR_INVALID
        assert L.sb_cvt_bgr_to_yuv420(fmt, dst.ctypes.data, 8, 8, 4, p, q) == SB_ERR_INVALID  # BGR pitch < 3 w
        assert L.sb_cvt_yuv420_to_bgr(fmt, (C.c_void_p * 3)(u8.ctypes.data), q, 8, 4, dst.ctypes.data, 64) == SB_ERR_INVALID
    assert L.sb_cvt_yuv420_to_bgr(0, p, q, 8, 4, dst.ctypes.data, 64) == SB_ERR_INVALID
    assert L.sb_cvt_yuv420_to_bgr(7, p, q, 8, 4, dst.ctypes.data, 64) == SB_ERR_INVALID
    with pytest.raises(StitchingError, match="even"):
        color.bgr_to_yuv420(np.zeros((4, 5, 3), np.uint8), "nv12")
    with pytest.raises(StitchingError, match="even"):
        color.yuv420_to_bgr(np.zeros((6, 5), np.uint8), "i420")

    # odd source frames (cfg 2 at 1/16: 250 x 187)
    cfg, cams, sizes, warper = small_rig("cfg2", 16, 2)
    c = Compositor(cams, sizes, warper, cfg["blender"], cfg["strength"])
    frame = np.zeros((cfg["h"] * 3 // 2, cfg["w"]), np.uint8)
    for fmt in ("nv12", "i420"):
        with pytest.raises(StitchingError, match="even"):
            c.upload([frame] * 2, fmt=fmt)
        with pytest.raises(StitchingError, match="even"):
            c.submit([frame] * 2, None, None, in_fmt=fmt)
    c.close()

    # an odd panorama (cfg 2 at 1/10: 400 x 300 sources, 1837 x 295 panorama): YUV in works, YUV out is refused
    cfg, cams, sizes, warper = small_rig("cfg2", 10, 2)
    c = Compositor(cams, sizes, warper, cfg["blender"], cfg["strength"])
    _, _, pw, ph = c.roi
    assert pw % 2 or ph % 2
    frames = [random_frame(cfg["w"], cfg["h"], "nv12", i) for i in range(2)]
    c.upload(frames, fmt="nv12")
    for fmt in ("nv12", "i420"):
        with pytest.raises(StitchingError, match="even"):
            c.download(fmt=fmt)
        with pytest.raises(StitchingError, match="even"):
            c.submit(frames, np.empty((ph * 3 // 2, pw), np.uint8), None, in_fmt="nv12", out_fmt=fmt)
    rc = L.sb_compositor_download_frame(c._c, 1, *planes(), None, 0)
    assert rc == SB_ERR_INVALID and b"even" in L.sb_last_error()
    c.close()

    # short pitches and missing planes through the compositor entries
    cfg, cams, sizes, warper = small_rig("cfg2", 20, 2)
    c = Compositor(cams, sizes, warper, cfg["blender"], cfg["strength"])
    w, h = cfg["w"], cfg["h"]
    _, _, pw, ph = c.roi
    buf = np.zeros((4 * max(h, ph), 4 * max(w, pw)), np.uint8)
    good_nv = ((C.c_void_p * 3)(buf.ctypes.data, buf.ctypes.data + h * w, None), (C.c_size_t * 3)(w, w, 0))
    assert L.sb_compositor_upload_frame(c._c, 0, 1, *good_nv, 0) == 0
    for k, short in ((0, w - 1), (1, w - 2)):
        pitches = (C.c_size_t * 3)(w, w, 0)
        pitches[k] = short
        assert L.sb_compositor_upload_frame(c._c, 0, 1, good_nv[0], pitches, 0) == SB_ERR_INVALID
    i420_short = (C.c_size_t * 3)(w, w // 2 - 1, w // 2)
    assert L.sb_compositor_upload_frame(c._c, 0, 2, (C.c_void_p * 3)(buf.ctypes.data, buf.ctypes.data, buf.ctypes.data), i420_short, 0) == SB_ERR_INVALID
    assert L.sb_compositor_upload_frame(c._c, 0, 2, good_nv[0], (C.c_size_t * 3)(w, w, w), 0) == SB_ERR_INVALID  # no V plane
    assert L.sb_compositor_upload_frame(c._c, 0, 3, *good_nv, 0) == SB_ERR_INVALID  # unknown format
    assert L.sb_compositor_upload_frame(c._c, 5, 1, *good_nv, 0) == SB_ERR_INVALID  # no such image
    out_p = (C.c_void_p * 3)(buf.ctypes.data, buf.ctypes.data, buf.ctypes.data)
    assert L.sb_compositor_download_frame(c._c, 1, out_p, (C.c_size_t * 3)(pw, pw - 1, 0), None, 0) == SB_ERR_INVALID
    assert L.sb_compositor_download_frame(c._c, 2, out_p, (C.c_size_t * 3)(pw, pw // 2, pw // 2 - 1), None, 0) == SB_ERR_INVALID
    assert L.sb_compositor_download_frame(c._c, 0, out_p, (C.c_size_t * 3)(3 * pw - 1, 0, 0), None, 0) == SB_ERR_INVALID
    assert L.sb_compositor_download_frame(c._c, 1, out_p, (C.c_size_t * 3)(pw, pw, 0), buf.ctypes.data, pw - 1) == SB_ERR_INVALID
    srcs = (C.c_void_p * 6)(*([buf.ctypes.data] * 6))
    ticket = C.c_ulonglong()
    assert L.sb_compositor_submit_frames(c._c, 1, srcs, (C.c_size_t * 6)(w, w, 0, w, w - 1, 0), 0, None, None, None, 0,
                                         C.byref(ticket)) == SB_ERR_INVALID
    assert L.sb_compositor_submit_frames(c._c, 1, srcs, (C.c_size_t * 6)(w, w, 0, w, w, 0), 1, out_p,
                                         (C.c_size_t * 3)(pw - 1, pw, 0), None, 0, C.byref(ticket)) == SB_ERR_INVALID
    assert L.sb_compositor_submit_frames(c._c, 1, srcs, (C.c_size_t * 6)(w, w, 0, w, w, 0), 4, None, None, None, 0,
                                         C.byref(ticket)) == SB_ERR_INVALID
    with pytest.raises(StitchingError):
        c.upload([np.zeros((h, w), np.uint8)] * 2, fmt="nv12")  # not (h * 3/2, w)
    with pytest.raises(StitchingError):
        c.upload([np.zeros((h * 3 // 2, w), np.uint8)] * 2, fmt="yuyv")
    with pytest.raises(StitchingError, match="C-contiguous"):
        c.download(out=np.zeros((ph * 3 // 2, 2 * pw), np.uint8)[:, :pw], fmt="i420")
    c.close()


def check_sharded_refuses_yuv():
    cfg, cams, sizes, warper = small_rig("cfg2", 20)
    c = Compositor(cams, sizes, warper, cfg["blender"], cfg["strength"], rank=0, world=2)
    L = _lib.lib()
    frame = random_frame(cfg["w"], cfg["h"], "nv12", 0)
    p, q, _ = color.planes(frame, cfg["w"], cfg["h"], "nv12")
    assert L.sb_compositor_upload_frame(c._c, 0, 1, p, q, 0) == SB_ERR_STATE
    assert b"single-GPU" in L.sb_last_error()
    h, w = c.roi[3], c.strip[1] - c.strip[0]
    out = np.empty((h * 3 // 2 + 2, w + 2), np.uint8)
    op, oq, _ = color.planes(out[: (h // 2) * 3, : w // 2 * 2], w // 2 * 2, h // 2 * 2, "nv12", writable=True)
    assert L.sb_compositor_download_frame(c._c, 1, op, oq, None, 0) == SB_ERR_STATE
    srcs = (C.c_void_p * (3 * len(cams)))()
    pitches = (C.c_size_t * (3 * len(cams)))()
    assert L.sb_compositor_submit_frames(c._c, 1, srcs, pitches, 1, None, None, None, 0, None) == SB_ERR_STATE
    with pytest.raises(StitchingError, match="single-GPU"):
        c.upload([frame] * c.count, fmt="nv12")
    c.close()


# ---- the oracle against cv2 and the golden data --------------------------------------------------------------------
def test_oracle_yuv_to_bgr_exhaustive_against_cv2():
    cv = pytest.importorskip("cv2")
    for fmt, code in (("nv12", cv.COLOR_YUV2BGR_NV12), ("i420", cv.COLOR_YUV2BGR_I420)):
        frame = YO.exhaustive_frame(fmt)
        Y, U, V = YO.split(frame, fmt)
        # every (Y, U, V) triple exactly once
        trip = (Y.astype(np.int64) << 16) | (np.repeat(np.repeat(U, 2, 0), 2, 1).astype(np.int64) << 8) | np.repeat(np.repeat(V, 2, 0), 2, 1)
        assert np.unique(trip).size == 1 << 24
        got, exp = YO.yuv420_to_bgr(frame, fmt), cv.cvtColor(frame, code)
        assert np.array_equal(got, exp), f"{fmt}: {int((got != exp).sum())} values differ from cv2"


def test_oracle_bgr_to_i420_against_cv2():
    cv = pytest.importorskip("cv2")
    sizes = [(2, 2), (4, 2), (2, 6), (10, 8), (34, 18), (1500, 1000)]
    for k, (w, h) in enumerate(sizes):
        img = random_frame(w, h, "bgr", 300 + k)
        assert np.array_equal(YO.bgr_to_yuv420(img, "i420"), cv.cvtColor(img, cv.COLOR_BGR2YUV_I420)), f"{w}x{h}"
    cube = np.array([[b, g, r] for b in (0, 255) for g in (0, 255) for r in (0, 255)], np.uint8)
    img = np.repeat(np.repeat(cube.reshape(2, 4, 3), 3, 0), 5, 1)[:6, :20]  # the corners, not block-aligned
    assert np.array_equal(YO.bgr_to_yuv420(img, "i420"), cv.cvtColor(img, cv.COLOR_BGR2YUV_I420))
    dark = np.random.default_rng(5).integers(0, 20, (64, 64, 3), dtype=np.uint8)  # Y < 16
    assert np.array_equal(YO.bgr_to_yuv420(dark, "i420"), cv.cvtColor(dark, cv.COLOR_BGR2YUV_I420))
    # NV12 output is the I420 result with U and V interleaved
    i420 = cv.cvtColor(img, cv.COLOR_BGR2YUV_I420)
    assert np.array_equal(YO.bgr_to_yuv420(img, "nv12"), YO.join(*YO.split(i420, "i420"), "nv12"))


def test_oracle_and_cv2_reject_odd_sizes():
    for w, h in ((5, 4), (4, 5), (3, 3)):
        with pytest.raises(ValueError):
            YO.bgr_to_yuv420(np.zeros((h, w, 3), np.uint8), "i420")
    for shape in ((6, 5), (7, 4)):  # an odd width; a height that is not a whole number of h * 3/2 rows
        for fmt in ("nv12", "i420"):
            with pytest.raises(ValueError):
                YO.yuv420_to_bgr(np.zeros(shape, np.uint8), fmt)
    cv = pytest.importorskip("cv2")
    with pytest.raises(cv.error):
        cv.cvtColor(np.zeros((4, 5, 3), np.uint8), cv.COLOR_BGR2YUV_I420)
    with pytest.raises(cv.error):
        cv.cvtColor(np.zeros((6, 5), np.uint8), cv.COLOR_YUV2BGR_NV12)


def test_oracle_reproduces_golden_cv2_results():
    z = np.load(GOLDEN)
    names = sorted({k.split("__")[0] for k in z.files})
    assert len(names) >= 10
    for name in names:
        kind, x, want = name.split("_")[0], z[name + "__in"], z[name + "__out"]
        got = YO.bgr_to_yuv420(x, "i420") if kind == "bgr" else YO.yuv420_to_bgr(x, kind)
        assert np.array_equal(got, want), name


# ---- the product's kernels through tests/emu -----------------------------------------------------------------------
def test_conversions_equal_oracle(use_emu):
    check_golden_through_library()
    check_random_conversions_through_library()


def test_conversions_of_the_exhaustive_frame(use_emu):
    check_exhaustive_frame_through_library()


def test_yuv_upload_equals_bgr_upload_of_the_oracle_frames(use_emu, monkeypatch):
    check_upload_equals_oracle_bgr_upload(monkeypatch)
    # a projection whose warp kernel reads the packed 3-byte sources even when word-per-pixel ones exist
    check_upload_equals_oracle_bgr_upload(monkeypatch, n=2, warper="fisheye")


def test_yuv_download_equals_oracle(use_emu):
    check_download_equals_oracle()


def test_submit_every_format_pair_equals_composite(use_emu):
    check_submit_all_format_pairs()


def test_bgr_calls_unchanged_next_to_yuv_calls(use_emu):
    """The BGR entries are the format-taking ones with SB_PIX_BGR: a BGR composite is the same before and after YUV use."""
    cfg, cams, sizes, warper = small_rig("cfg2", 20, 3)
    c = Compositor(cams, sizes, warper, cfg["blender"], cfg["strength"])
    imgs = [rigs.noise_image(cfg["h"], cfg["w"], 7 + i) for i in range(len(cams))]
    p0, m0 = (a.copy() for a in c.composite(imgs))
    c.composite([YO.bgr_to_yuv420(im, "i420") for im in imgs], in_fmt="i420", out_fmt="nv12")
    p1, m1 = c.composite(imgs)
    assert np.array_equal(p0, p1) and np.array_equal(m0, m1)
    c.close()


def test_error_cases(use_emu):
    check_error_cases()


def test_sharded_compositor_refuses_yuv(use_emu):
    check_sharded_refuses_yuv()
