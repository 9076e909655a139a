"""Replay of the committed golden vectors (tests/golden/*.npz) against an implementation.

The same functions check the CPU oracle (tests/test_oracle_golden.py) and the CUDA path through the Python
drop-ins (tests/test_gpu_parity.py, tests/test_host_logic.py via the emulation build).
"""
import hashlib
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load(name):
    return np.load(os.path.join(GOLDEN, name), allow_pickle=False)


def diff_report(got, exp, what):
    got = np.asarray(got)
    exp = np.asarray(exp)
    assert got.shape == exp.shape, f"{what}: shape {got.shape} != {exp.shape}"
    d = np.abs(got.astype(np.int64) - exp.astype(np.int64))
    n = int((d != 0).sum())
    return n, (int(d.max()) if n else 0), f"{what}: {n}/{d.size} values differ, max |diff| {int(d.max()) if d.size else 0}"


def assert_exact(got, exp, what):
    n, mx, msg = diff_report(got, exp, what)
    assert n == 0, msg


PACK_WHOLE_BYTES = 2048  # larger arrays are stored as shape + sha256 + a sample, so that a golden file stays small
PACK_SAMPLE = 64


def _sample_index(size):
    return np.sort(np.random.default_rng(size).choice(size, min(size, PACK_SAMPLE), replace=False))


def pack(out, key, arr):
    """Store the expected array `arr` under `key` in the dict `out` (later np.savez_compressed): whole when small, else one
    string "dtype shape sha256 sample" -- the sha256 of all its values and, in hex, a fixed sample of them (for the report
    when they differ)."""
    arr = np.ascontiguousarray(arr)
    if arr.nbytes <= PACK_WHOLE_BYTES:
        out[key] = arr
        return
    sample = arr.reshape(-1)[_sample_index(arr.size)]
    out[f"{key}__digest"] = np.bytes_(" ".join([str(arr.dtype), "x".join(str(d) for d in arr.shape), hashlib.sha256(arr.tobytes()).hexdigest(),
                                                sample.tobytes().hex()]))


def assert_golden(got, g, key, what):
    """`got` equals, value for value, the array pack() stored under `key` in the loaded golden file `g`."""
    if key in g.files:
        assert_exact(got, g[key], what)
        return
    dtype, shape, sha, sample = g[f"{key}__digest"].item().decode().split(" ")
    got = np.ascontiguousarray(got)
    shape = tuple(int(d) for d in shape.split("x"))
    assert got.shape == shape, f"{what}: shape {got.shape} != {shape}"
    assert str(got.dtype) == dtype, f"{what}: dtype {got.dtype} != {dtype}"
    assert_exact(got.reshape(-1)[_sample_index(got.size)], np.frombuffer(bytes.fromhex(sample), dtype), f"{what} (sampled values)")
    assert hashlib.sha256(got.tobytes()).hexdigest() == sha, f"{what}: the sampled values agree, but not all {got.size} values (sha256 differs)"


def warp_cases():
    """The warped image and mask of case i are stored with pack() under img_<i> / mask_<i> of `g`; the sources are drawn
    again from the generator's seed (tests/golden/gen_golden.py gen_warp) and checked against the recorded sha256."""
    g = load("golden_warp.npz")
    from stitching_b200 import rigs

    rng = np.random.default_rng(20260922)
    srcs = [rng.integers(0, 256, (72, 96, 3), dtype=np.uint8) for _ in range(int(g["n"]))]
    h = hashlib.sha256()
    for src in srcs:
        h.update(src.tobytes())
    assert h.hexdigest() == str(g["src_sha256"]), "the seeded warp sources drifted from the goldens"
    for i, src in enumerate(srcs):
        f, a, px, py = g[f"cam_{i}"]
        cam = rigs.Camera(f, a, px, py, g[f"R_{i}"])
        yield dict(i=i, wtype=str(g[f"type_{i}"]), cam=cam, scale=float(g[f"scale_{i}"]), aspect=float(g[f"aspect_{i}"]),
                   src=src, roi=tuple(int(v) for v in g[f"roi_{i}"]), g=g)


def blend_cases():
    g = load("golden_blend.npz")
    for i in range(int(g["n"])):
        n = int(g[f"count_{i}"])
        yield dict(i=i, btype=str(g[f"type_{i}"]), strength=float(g[f"strength_{i}"]),
                   imgs=[g[f"img_{i}_{j}"] for j in range(n)], masks=[g[f"mask_{i}_{j}"] for j in range(n)],
                   corners=[tuple(int(v) for v in g[f"corner_{i}_{j}"]) for j in range(n)],
                   pano=g[f"pano_{i}"], pmask=g[f"pmask_{i}"])


def e2e_cases():
    g = load("golden_e2e.npz")
    from stitching_b200 import rigs

    for name in ("cfg2", "cfg3", "cfg5"):
        cfg = rigs.config(name, int(g[f"{name}_scale_down"]))
        n = int(g[f"{name}_n"])
        cams = cfg["cameras"][:n]
        imgs = [rigs.synth_image(cfg["h"], cfg["w"], i) for i in range(n)]
        h = hashlib.sha256()
        for im in imgs:
            h.update(im.tobytes())
        assert h.hexdigest() == str(g[f"{name}_input_sha256"]), "synthetic input generator drifted from the goldens"
        yield dict(name=name, cfg=cfg, cams=cams, imgs=imgs, corners=[tuple(int(v) for v in r) for r in g[f"{name}_corners"]],
                   sizes=[tuple(int(v) for v in r) for r in g[f"{name}_sizes"]], g=g)  # pano / pmask: <name>_pano, <name>_pmask (pack)


def run_warper_goldens(WarperCls):
    """WarperCls follows stitching/warper.py's interface."""
    for c in warp_cases():
        w = WarperCls(c["wtype"])
        w.scale = c["scale"]
        size = (c["src"].shape[1], c["src"].shape[0])
        assert tuple(w.warp_roi(size, c["cam"], c["aspect"])) == c["roi"], f"warp case {c['i']} ({c['wtype']}): roi"
        assert_golden(w.warp_image(c["src"], c["cam"], c["aspect"]), c["g"], f"img_{c['i']}", f"warp case {c['i']} ({c['wtype']}) image")
        assert_golden(w.create_and_warp_mask(size, c["cam"], c["aspect"]), c["g"], f"mask_{c['i']}", f"warp case {c['i']} ({c['wtype']}) mask")


def run_blender_goldens(BlenderCls):
    """BlenderCls follows stitching/blender.py's interface."""
    for c in blend_cases():
        b = BlenderCls(c["btype"], c["strength"])
        sizes = [(m.shape[1], m.shape[0]) for m in c["masks"]]
        b.prepare(c["corners"], sizes)
        for img, m, corner in zip(c["imgs"], c["masks"], c["corners"]):
            b.feed(img, m, corner)
        pano, pmask = b.blend()
        assert_exact(pano, c["pano"], f"blend case {c['i']} ({c['btype']} strength {c['strength']}) pano")
        assert_exact(pmask, c["pmask"], f"blend case {c['i']} ({c['btype']}) mask")


def run_e2e_goldens(WarperCls, BlenderCls):
    for c in e2e_cases():
        cfg = c["cfg"]
        w = WarperCls(cfg["warper"])
        w.set_scale(c["cams"])
        sizes_in = [(cfg["w"], cfg["h"])] * len(c["cams"])
        warped = list(w.warp_images(c["imgs"], c["cams"]))
        masks = list(w.create_and_warp_masks(sizes_in, c["cams"]))
        corners, sizes = w.warp_rois(sizes_in, c["cams"])
        assert [tuple(x) for x in corners] == c["corners"] and [tuple(x) for x in sizes] == c["sizes"], f"{c['name']}: rois"
        b = BlenderCls(cfg["blender"], cfg["strength"])
        b.prepare(corners, sizes)
        for img, m, corner in zip(warped, masks, corners):
            b.feed(img, m, corner)
        pano, pmask = b.blend()
        assert_golden(pano, c["g"], f"{c['name']}_pano", f"{c['name']} pano")
        assert_golden(pmask, c["g"], f"{c['name']}_pmask", f"{c['name']} mask")


class OracleWarper:
    """stitching/warper.py's interface on the CPU oracle (for the replay functions above)."""

    def __init__(self, wtype):
        from oracle import oracle as O
        from stitching_b200.warper import Warper

        self.O, self.wtype, self.scale, self._get_K = O, wtype, None, Warper.get_K

    def set_scale(self, cameras):
        from statistics import median

        self.scale = median([c.focal for c in cameras])

    def warp_roi(self, size, cam, aspect=1):
        return self.O.warp_roi(self.wtype, self.scale * aspect, self._get_K(cam, aspect), cam.R, size)

    def warp_image(self, img, cam, aspect=1):
        return self.O.warp(self.wtype, self.scale * aspect, self._get_K(cam, aspect), cam.R, img, True, False)[1]

    def create_and_warp_mask(self, size, cam, aspect=1):
        dummy = np.zeros((size[1], size[0], 3), np.uint8)
        return self.O.warp(self.wtype, self.scale * aspect, self._get_K(cam, aspect), cam.R, dummy, False, True)[2]

    def warp_images(self, imgs, cams, aspect=1):
        return (self.warp_image(i, c, aspect) for i, c in zip(imgs, cams))

    def create_and_warp_masks(self, sizes, cams, aspect=1):
        return (self.create_and_warp_mask(s, c, aspect) for s, c in zip(sizes, cams))

    def warp_rois(self, sizes, cams, aspect=1):
        rois = [self.warp_roi(s, c, aspect) for s, c in zip(sizes, cams)]
        return [r[0:2] for r in rois], [r[2:4] for r in rois]


def ramp_masks(masks, ramp=64):
    """Mask set B of SURVEY 8(d): the validity mask with a linear gray ramp toward the left/right neighbours
    (mimics SeamFinder.resize's 256-level output)."""
    out = []
    for m in masks:
        h, w = m.shape
        x = np.arange(w)
        r = np.minimum(np.minimum(x, w - 1 - x) * 255 // max(ramp, 1), 255).astype(np.uint8)
        out.append(np.minimum(m, r[None, :]))
    return out


def oracle_composite(O, cfg, cams, imgs, mask_fn=None):
    """Warp + blend on the CPU oracle the way stitcher.py:178-189, 241-259 drive the reference classes."""
    w = OracleWarper(cfg["warper"])
    w.set_scale(cams)
    warped, masks, corners, sizes = [], [], [], []
    for img, cam in zip(imgs, cams):
        rect, wi, wm = O.warp(cfg["warper"], w.scale, w._get_K(cam, 1), cam.R, img)
        warped.append(wi)
        masks.append(wm)
        corners.append(rect[:2])
        sizes.append(rect[2:])
    if mask_fn is not None:
        masks = mask_fn(masks)
    b = O.Blender(cfg["blender"], cfg["strength"])
    b.prepare(corners, sizes)
    for wi, wm, c in zip(warped, masks, corners):
        b.feed(wi, wm, c)
    pano, pmask = b.blend()
    return dict(warped=warped, masks=masks, corners=corners, sizes=sizes, pano=pano, pmask=pmask, num_bands=b.num_bands)


def run_seam_goldens(resize_fn):
    """SeamFinder.resize goldens (tests/golden/golden_seam.npz, written by the reference function)."""
    g = load("golden_seam.npz")
    for i in range(int(g["n"])):
        assert_exact(np.asarray(resize_fn(g[f"seam_{i}"], g[f"mask_{i}"])), g[f"out_{i}"], f"SeamFinder.resize case {i}")


def seam_masks_low(ref_masks, ratio=3.17, seed=0):
    """LOW-resolution seam masks for warped masks of a rig: a ragged seam through the middle of each (test input)."""
    rng = np.random.default_rng(seed)
    out = []
    for i, m in enumerate(ref_masks):
        h, w = m.shape
        sh, sw = max(2, int(round(h / ratio)) + i % 2), max(2, int(round(w / ratio)) - i % 3)
        s = np.zeros((sh, sw), np.uint8)
        s[:, : sw // 2 + int(rng.integers(-3, 4))] = 255
        ys = rng.integers(0, sh, 8)
        for y in ys:
            s[max(0, y - 2) : y + 3, sw // 2 - 4 : sw // 2 + 5] = 255 * int(rng.integers(0, 2))
        out.append(s if i % 2 else 255 - s)
    return out


def run_resize_goldens(resize_fn):
    """Images.resize_img_by_scaler goldens (tests/golden/golden_resize.npz): resize_fn(img, (w, h)) -> image."""
    g = load("golden_resize.npz")
    for i in range(int(g["n"])):
        size = tuple(int(v) for v in g[f"size_{i}"])
        assert_exact(np.asarray(resize_fn(g[f"img_{i}"], size)), g[f"out_{i}"], f"Images.resize case {i} -> {size}")


def run_timelapse_goldens(timelapser_cls):
    """Timelapser goldens (tests/golden/golden_timelapse.npz): initialize / process_frame / get_frame per image."""
    g = load("golden_timelapse.npz")
    for k in range(int(g["n"])):
        kind = str(g[f"kind_{k}"])
        corners = [tuple(int(v) for v in c) for c in g[f"corners_{k}"]]
        sizes = [tuple(int(v) for v in s) for s in g[f"sizes_{k}"]]
        t = timelapser_cls(kind)
        t.initialize(corners, sizes)
        for i, c in enumerate(corners):
            t.process_frame(g[f"img_{k}_{i}"], c)
            assert_exact(np.asarray(t.get_frame()), g[f"frame_{k}_{i}"], f"timelapse case {k} ({kind}) frame {i}")


def timelapse_fuzz(oracle, timelapser_cls, warper_cls, rigs, scale_down, seed=77):
    """Random rects against the oracle's restatement, int16 inputs included, and -- the pipeline's case -- frames fed from
    warped images that still have their device twin (stitcher.py:249-252 hands Timelapser the warper's output)."""
    rng = np.random.default_rng(seed)
    for t in range(6):
        kind = "as_is" if t % 2 == 0 else "crop"
        n = int(rng.integers(2, 5))
        sizes = [(int(rng.integers(30, 300)), int(rng.integers(20, 200))) for _ in range(n)]
        corners = [(int(rng.integers(-40, 40)) + 25 * i, int(rng.integers(-30, 30))) for i in range(n)]
        a, b = timelapser_cls(kind), oracle.Timelapser(kind)
        a.initialize(corners, sizes)
        b.initialize(corners, sizes)
        for i, ((w, h), c) in enumerate(zip(sizes, corners)):
            img = rigs.noise_image(h, w, 50 * t + i)
            if t >= 4:
                img = (img.astype(np.int32) * 300 - 38000).clip(-32768, 32767).astype(np.int16)
            a.process_frame(img, c)
            b.process_frame(img, c)
            assert_exact(np.asarray(a.get_frame()), b.get_frame(), f"timelapse fuzz {t} ({kind}) frame {i}")
    cfg = rigs.config("cfg2", scale_down)
    cams = cfg["cameras"][1:4]
    w = warper_cls(cfg["warper"])
    w.set_scale(cams)
    sizes = [(cfg["w"], cfg["h"])] * len(cams)
    imgs = [rigs.synth_image(cfg["h"], cfg["w"], 9 + i) for i in range(len(cams))]
    warped = list(w.warp_images(imgs, cams))
    corners, wsizes = w.warp_rois(sizes, cams)
    for kind in ("as_is", "crop"):
        a, b = timelapser_cls(kind), oracle.Timelapser(kind)
        a.initialize(corners, wsizes)
        b.initialize(corners, wsizes)
        for i, (img, c) in enumerate(zip(warped, corners)):
            a.process_frame(img, c)               # device twin
            b.process_frame(np.array(img), c)     # plain host copy through the oracle
            assert_exact(np.asarray(a.get_frame()), b.get_frame(), f"timelapse of warped image {i} ({kind})")
            a.process_frame(img[3:-2, 5:-4], (c[0] + 5, c[1] + 3))  # a cropped view keeps the twin (cropper.py:150-151)
            b.process_frame(np.array(img[3:-2, 5:-4]), (c[0] + 5, c[1] + 3))
            assert_exact(np.asarray(a.get_frame()), b.get_frame(), f"timelapse of cropped warped image {i} ({kind})")


def run_gain_goldens(apply_fn):
    """ExposureErrorCompensator.apply goldens (tests/golden/golden_gain.npz): apply_fn(img, gain) -> image."""
    g = load("golden_gain.npz")
    for i in range(int(g["n"])):
        gain = g[f"gain_{i}"]
        got = g[f"img_{i}"] if gain.size == 0 else np.asarray(apply_fn(g[f"img_{i}"], gain))  # compensator "no": identity
        assert_exact(got, g[f"out_{i}"], f"compensator apply case {i} ({g[f'kind_{i}']})")


def fused_chain_case(oracle, Warper, Blender, Compositor, rigs, scale_down):
    """The whole FINAL-resolution chain fused in the compositor -- warp, exposure gain, seam mask, blend -- against the
    reference order of operations with the drop-in classes and the oracle's apply / SeamFinder.resize in between
    (stitcher.py:219-225, 254)."""
    cfg = rigs.config("cfg2", scale_down)
    cams = cfg["cameras"]
    n = len(cams)
    sizes_in = [(cfg["w"], cfg["h"])] * n
    imgs = [rigs.noise_image(cfg["h"], cfg["w"], 90 + i) if i % 2 else rigs.synth_image(cfg["h"], cfg["w"], 90 + i) for i in range(n)]
    rng = np.random.default_rng(19)
    gains = [rng.uniform(0.75, 1.4, (4 + i % 3, 6)).astype(np.float32) if i % 3 else None for i in range(n)]  # some images without
    w = Warper(cfg["warper"])
    w.set_scale(cams)
    corners, sizes = w.warp_rois(sizes_in, cams)
    warped = [w.warp_image_and_mask(imgs[i], cams[i]) for i in range(n)]
    seams = seam_masks_low([m for _, m in warped], seed=3)
    b = Blender(cfg["blender"], cfg["strength"])
    b.prepare(corners, sizes)
    for i in range(n):
        wi, wm = warped[i]
        if gains[i] is not None:
            wi = oracle.gain_apply(wi, gains[i])
        b.feed(wi, oracle.seam_resize(seams[i], wm) if i != 1 else wm, corners[i])  # image 1 keeps its validity mask
    ref = b.blend()
    c = Compositor(cams, sizes_in, cfg["warper"], cfg["blender"], cfg["strength"])
    for i in range(n):
        c.set_gain(i, gains[i])
        if i != 1:
            c.set_seam_mask(i, seams[i])
    got = c.composite(imgs)
    c.close()
    return got, ref


def fused_gain_case(oracle, Warper, Blender, Compositor, rigs, scale_down, kinds=("gain_blocks", "channel_blocks", "gain", "channel")):
    """Compositor.set_gain (gain applied in the warp kernel) against the reference order of operations done with the
    drop-in classes and the ORACLE's apply in between: warp -> ExposureErrorCompensator.apply -> Blender.feed
    (stitcher.py:219-221, 254).  One synthetic gain of each kind, cycling over the images."""
    cfg = rigs.config("cfg2", scale_down)
    cams = cfg["cameras"]
    n = len(cams)
    sizes_in = [(cfg["w"], cfg["h"])] * n
    imgs = [rigs.synth_image(cfg["h"], cfg["w"], 80 + i) for i in range(n)]
    rng = np.random.default_rng(17)
    gains = []
    for i in range(n):
        kind = kinds[i % len(kinds)]
        if kind == "gain_blocks":
            gains.append(rng.uniform(0.7, 1.5, (5 + i, 7)).astype(np.float32))
        elif kind == "channel_blocks":
            gains.append(rng.uniform(0.7, 1.5, (4, 6 + i, 3)).astype(np.float32))
        elif kind == "gain":
            gains.append(np.array([[rng.uniform(0.7, 1.5)]], np.float64))
        else:
            gains.append(np.array([[rng.uniform(0.7, 1.5)], [rng.uniform(0.7, 1.5)], [rng.uniform(0.7, 1.5)], [0.0]], np.float64))
    w = Warper(cfg["warper"])
    w.set_scale(cams)
    corners, sizes = w.warp_rois(sizes_in, cams)
    b = Blender(cfg["blender"], cfg["strength"])
    b.prepare(corners, sizes)
    for i in range(n):
        wi, wm = w.warp_image_and_mask(imgs[i], cams[i])
        b.feed(oracle.gain_apply(wi, gains[i]), wm, corners[i])
    ref_pano, ref_mask = b.blend()
    c = Compositor(cams, sizes_in, cfg["warper"], cfg["blender"], cfg["strength"])
    for i in range(n):
        c.set_gain(i, gains[i])
    pano, mask = c.composite(imgs)
    c.set_gain(0, None)  # and it can be removed again
    pano0, _ = c.composite(imgs)
    c.close()
    return (pano, mask), (ref_pano, ref_mask), pano0
