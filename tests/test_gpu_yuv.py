"""YUV 4:2:0 frames (NV12 / I420) in and out of the compositor on the B200: the checks of tests/test_yuv.py through the
CUDA kernels (sb_yuv.cu), and the full-size cfg 2 composite with NV12 in and out against the oracle chain."""
import numpy as np
import pytest

import test_yuv as T
import yuv_oracle as YO
from stitching_b200 import Compositor, StitchingError, rigs

pytestmark = pytest.mark.gpu


def test_conversions_equal_oracle_on_gpu(cuda_lib):
    T.check_golden_through_library()
    T.check_random_conversions_through_library()


def test_exhaustive_frame_through_the_kernels(cuda_lib):
    T.check_exhaustive_frame_through_library()


@pytest.mark.parametrize("name,scale_down,n,warper", [("cfg2", 20, None, None), ("cfg3", 10, 8, None), ("cfg2", 20, 3, "fisheye")])
def test_yuv_upload_equals_bgr_upload_on_gpu(cuda_lib, monkeypatch, name, scale_down, n, warper):
    T.check_upload_equals_oracle_bgr_upload(monkeypatch, name, scale_down, n, warper)


def test_yuv_download_equals_oracle_on_gpu(cuda_lib):
    T.check_download_equals_oracle()
    T.check_download_equals_oracle("cfg3", 10, 8)


def test_submit_every_format_pair_on_gpu(cuda_lib):
    T.check_submit_all_format_pairs(steps=3)


def test_error_cases_on_gpu(cuda_lib):
    T.check_error_cases()
    T.check_sharded_refuses_yuv()


def test_full_size_cfg2_nv12_to_nv12(cuda_lib):
    """BASELINE cfg 2 at full size (8 x 4000x3000 spherical, multiband): NV12 frames in, NV12 panorama out, through the
    pipelined path and the synchronous one, against the oracle chain -- the BGR composite of the oracle-converted frames,
    converted back by the oracle: 0 differing values."""
    cfg = rigs.config("cfg2", 1)
    cams = cfg["cameras"]
    w, h = cfg["w"], cfg["h"]
    c = Compositor(cams, [(w, h)] * len(cams), cfg["warper"], cfg["blender"], cfg["strength"])
    _, _, pw, ph = c.roi
    frames = [YO.bgr_to_yuv420(rigs.synth_image(h, w, i) if i % 2 else rigs.noise_image(h, w, 40 + i), "nv12") for i in range(len(cams))]
    bgr_pano, bgr_mask = (a.copy() for a in c.composite([YO.yuv420_to_bgr(f, "nv12") for f in frames]))
    expected = YO.bgr_to_yuv420(bgr_pano, "nv12")
    pano, mask = c.composite(frames, in_fmt="nv12", out_fmt="nv12")
    d = pano != expected
    assert not d.any(), f"{int(d.sum())} of {d.size} values differ"
    assert np.array_equal(mask, bgr_mask)
    pinned = [c.pinned_empty(f.shape) for f in frames]
    for p, f in zip(pinned, frames):
        p[...] = f
    out = c.pinned_empty((ph * 3 // 2, pw))
    c.wait(c.submit(pinned, out, None, in_fmt="nv12", out_fmt="nv12"))
    assert np.array_equal(out, expected)
    c.close()


def test_full_size_cfg5_panorama_is_refused_as_yuv(cuda_lib):
    """cfg 5's panorama (6544 x 4937) has an odd height: NV12 / I420 output is refused, as cv2 refuses it."""
    cfg = rigs.config("cfg5", 1)
    c = Compositor(cfg["cameras"], [(cfg["w"], cfg["h"])] * cfg["n"], cfg["warper"], cfg["blender"], cfg["strength"])
    assert c.roi[2:] == (6544, 4937)
    for fmt in ("nv12", "i420"):
        with pytest.raises(StitchingError, match="even"):
            c.download(fmt=fmt)
    c.close()
