#!/usr/bin/env python
"""bench.py -- warp + multiband-blend throughput of the B200 compositing path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload cfg2] [--dump-outputs DIR]

`--dump-outputs DIR` (--impl ours, one GPU or --replicas) writes what the last timed step computed, see dump_outputs().

One "step" = one pass of the hot path over one batch of synthetic frames for a fixed rig: fused warp of
every image (+ validity mask), Gaussian/weight pyramids, per-band weighted accumulate + normalise + collapse,
final uint8 panorama + mask.  At N = 1 the workload is BASELINE.json configs[1] (8 x 4000x3000 RGB, spherical
warp, multiband blend).  With N > 1 (torchrun, one rank per GPU) the ranks composite ONE panorama of the
BASELINE configs[2] family (4 images of 4000x3000 per GPU, cylindrical; N = 8 is configs[2] itself): image blocks
and pano column strips per rank, one grouped NCCL send/recv of the per-band partial sums (weak scaling);
`--replicas` runs one independent configs[1] panorama per GPU instead.

Prints ONE JSON line (rank 0).  `value` is device-resident throughput (inputs already in HBM, CUDA events on
the launching stream); `e2e` goes through the public API with pinned HOST buffers, host<->device copies inside
the timed region; `roofline` is the dominant kernel against the measured HBM copy bandwidth; `cpu_baseline`
is the reference's own cv2 path (oracle/cv_path.py) timed on this box's host cores.
"""
import argparse
import ctypes as C
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "warp+multiband-blend input MPix/s"
UNIT = "MPix/s"

WORKLOADS = {
    "cfg2": "8x4000x3000 RGB, spherical warp + multiband blend (BASELINE configs[1])",
    "cfg4": "8x8000x6000 RGB, spherical warp + multiband blend (BASELINE configs[3])",
    "cfg3": "32x4000x3000 RGB, cylindrical warp + multiband blend (BASELINE configs[2], all on one GPU)",
    "cfg5": "16x2000x1500 RGB, affine warp + feather blend (BASELINE configs[4])",
}


def dist_env():
    return int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))


class Dist:
    """torch.distributed (gloo) for the barrier and the max-over-ranks; only plumbing."""

    def __init__(self, world):
        self.world = world
        self.pg = None
        if world > 1:
            import torch.distributed as dist

            dist.init_process_group(backend="gloo")
            self.pg = dist

    def barrier(self):
        if self.pg:
            self.pg.barrier()

    def max(self, v):
        if not self.pg:
            return v
        import torch

        t = torch.tensor([float(v)], dtype=torch.float64)
        self.pg.all_reduce(t, op=self.pg.ReduceOp.MAX)
        return float(t.item())

    def sum(self, v):
        if not self.pg:
            return v
        import torch

        t = torch.tensor([float(v)], dtype=torch.float64)
        self.pg.all_reduce(t, op=self.pg.ReduceOp.SUM)
        return float(t.item())

    def close(self):
        if self.pg:
            self.pg.destroy_process_group()


class ClockSampler(threading.Thread):
    """SM clock + throttle reasons of one GPU sampled with NVML while the timed region runs."""

    def __init__(self, index, period=0.02):
        super().__init__(daemon=True)
        self.index, self.period, self.samples, self.reasons, self.stop_flag = index, period, [], set(), False
        self.max_mhz = None
        self.ok = False
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception as e:  # noqa: BLE001
            self.err = str(e)

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:  # noqa: BLE001
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:  # noqa: BLE001
                pass
            time.sleep(self.period)

    def result(self):
        self.stop_flag = True
        if self.ok:
            self.join(timeout=1)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0,
                    "note": getattr(self, "err", "no sample landed inside the timed region")}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:  # noqa: BLE001
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic(kernel):
    """DRAM bytes per launch of `kernel` from the committed ncu capture, if one exists for this round."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)).get(kernel)
        except Exception:  # noqa: BLE001
            return None
    return None


SCALE_DOWN = 1  # --scale-down (debug dry runs only; recorded in config, never a reportable number)


def make_workload(name, rank):
    from stitching_b200 import rigs

    cfg = rigs.config(name, SCALE_DOWN)
    imgs = [rigs.synth_image(cfg["h"], cfg["w"], 100 * rank + i) for i in range(cfg["n"])]
    return cfg, imgs


def cpu_reference_run(cfg, imgs, n_sample, threads=None, want_result=False):
    """One pass of the reference's CPU path over the first n_sample images of the ring (n_sample = cfg['n']: the whole
    configuration).  Returns (MPix/s, seconds, info[, pano, mask])."""
    from oracle import cv_path

    cams = cfg["cameras"][:n_sample]
    sub = imgs[:n_sample]
    mpix = sum(im.shape[0] * im.shape[1] for im in sub) / 1e6
    if cv_path.available():
        t0 = time.perf_counter()
        pano, mask, stages = cv_path.composite(cfg, cams, sub, threads)
        dt = time.perf_counter() - t0
        info = cv_path.describe()
        out = (mpix / dt, dt, {"backend": f"cv2 {info['cv2']}", "cores": info["threads"], "parallel": info["parallel"],
                               "stages_s": {k: round(v, 3) for k, v in stages.items()}})
        if want_result:
            if hasattr(mask, "get"):
                mask = mask.get()
            return out + (pano, mask)
        return out
    # cv2 missing on this box: the scalar C restatement (1 core)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import replay
    from oracle import oracle as O

    t0 = time.perf_counter()
    ref = replay.oracle_composite(O, cfg, cams, sub)
    dt = time.perf_counter() - t0
    out = (mpix / dt, dt, {"backend": "oracle/stitch_oracle.c (scalar)", "cores": 1, "parallel": "", "stages_s": {}})
    return out + (ref["pano"], ref["pmask"]) if want_result else out


def compare_results(pano, mask, ref_pano, ref_mask):
    """GPU result vs the CPU reference result of the same inputs: differing values and the largest difference."""
    if pano.shape != ref_pano.shape or mask.shape != ref_mask.shape:
        return {"shape_mismatch": [list(pano.shape), list(ref_pano.shape)]}
    differing, max_abs = 0, 0
    rows = 512
    for y in range(0, pano.shape[0], rows):  # in bands: the int16 temporaries of a 160 MB panorama stay small
        d = np.abs(pano[y:y + rows].astype(np.int16) - ref_pano[y:y + rows].astype(np.int16))
        differing += int(np.count_nonzero(d))
        max_abs = max(max_abs, int(d.max()) if d.size else 0)
    mask_diff = int(np.count_nonzero(mask != ref_mask))
    return {"differing": differing, "max_abs": max_abs, "mask_differing": mask_diff, "values": int(pano.size),
            "against": "the reference's cv2 path on the same inputs (oracle/cv_path.py), whole panorama"}


def cpu_baseline_block(cfg, imgs, gpu_pano=None, gpu_mask=None, budget_s=100.0):
    """BASELINE.md section 3: the WHOLE configuration through the reference's CPU path on this box's host cores, with
    all cores (one warm-up + up to 3 timed repetitions, median) and with one core (one repetition, as the time budget
    of a default bench run allows), plus the comparison of the GPU panorama with the CPU panorama."""
    n = cfg["n"]
    ncpu = os.cpu_count() or 1
    t_start = time.perf_counter()
    _, warm_dt, info, pano, mask = cpu_reference_run(cfg, imgs, n, threads=ncpu, want_result=True)
    parity = None
    if gpu_pano is not None:
        parity = compare_results(gpu_pano, gpu_mask, pano, mask)
    del pano, mask
    times = []
    reps = 3 if warm_dt * 3.2 < budget_s * 0.6 else 1
    for _ in range(reps):
        _, dt, info = cpu_reference_run(cfg, imgs, n, threads=ncpu)
        times.append(dt)
    mpix = n * cfg["w"] * cfg["h"] / 1e6
    med = float(np.median(times))
    block = {"value": mpix / med, "unit": UNIT, "cores": info["cores"], "kind": "port",
             "sample": f"the whole configuration ({n} images at full resolution) per repetition: 1 warm-up + {reps} timed, median "
                       f"{med:.2f} s, min {min(times):.2f} s ({info['backend']}, cv.setNumThreads({ncpu}); {info['parallel']})",
             "stages_s": info["stages_s"], "host_cpus": ncpu, "warmup_s": round(warm_dt, 2), "reps_s": [round(t, 2) for t in times]}
    # one core, if the remaining budget allows (the single-core pass of cfg 2 takes ~30-60 s)
    left = budget_s - (time.perf_counter() - t_start)
    if left > 45:
        v1, dt1, _ = cpu_reference_run(cfg, imgs, n, threads=1)
        block["one_core"] = {"value": v1, "unit": UNIT, "cores": 1, "seconds": round(dt1, 2), "sample": "the whole configuration, 1 cold repetition"}
    else:
        block["one_core"] = None
    return block, parity


def sharded_workload_name(n, w, h, world):
    return (f"cfg3 family: {n}x{w}x{h} RGB, cylindrical warp + multiband blend, ONE panorama sharded over {world} GPUs "
            f"(4 images per GPU; N=8 is BASELINE configs[2])" + (f" SCALED DOWN x{SCALE_DOWN} (debug)" if SCALE_DOWN != 1 else ""))


def run_reference(args, rank, world):
    if rank != 0:
        return
    if world > 1:  # the sharded arm's workload (run_sharded): 4 images per GPU on a cylindrical ring
        from stitching_b200 import rigs

        n, w, h = 4 * world, 4000 // SCALE_DOWN, 3000 // SCALE_DOWN
        cfg = dict(n=n, w=w, h=h, warper="cylindrical", cameras=rigs.yaw_ring(n, w, h, 8000 / SCALE_DOWN, 10), blender="multiband", strength=5)
        imgs = [rigs.synth_image(h, w, i) for i in range(n)]
        workload = sharded_workload_name(n, w, h, world)
    else:
        cfg, imgs = make_workload(args.workload, 0)
        workload = f"{args.workload}: {WORKLOADS[args.workload]}"
    ncpu = os.cpu_count() or 1
    # the whole configuration per step with all host cores; only if that cannot finish the requested steps within a few
    # minutes the step shrinks to the first images of the ring (and says so)
    n_sample = min(args.cpu_sample or cfg["n"], cfg["n"])
    v, dt, info = cpu_reference_run(cfg, imgs, n_sample, threads=ncpu)  # first (cold) pass = first warm-up step
    budget = 330.0
    while n_sample > 2 and dt * (args.steps + args.warmup) > budget:
        n_sample = max(2, n_sample // 2)
        v, dt, info = cpu_reference_run(cfg, imgs, n_sample, threads=ncpu)
    for _ in range(max(0, args.warmup - 1)):
        cpu_reference_run(cfg, imgs, n_sample, threads=ncpu)
    times = []
    for _ in range(args.steps):
        _, dt, info = cpu_reference_run(cfg, imgs, n_sample, threads=ncpu)
        times.append(dt)
    mpix = n_sample * cfg["w"] * cfg["h"] / 1e6
    value = mpix * len(times) / sum(times)
    whole = n_sample == cfg["n"]
    sample = (f"the whole configuration ({cfg['n']} images at full resolution) per step" if whole else
              f"first {n_sample} of {cfg['n']} images of the ring at full resolution per step (bounded: the whole ring would not finish "
              f"{args.steps + args.warmup} steps within a few minutes)") + f" ({info['backend']}, cv.setNumThreads({ncpu}))"
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * sum(times) / len(times), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "int16+f32 (uint8 in/out)", "data": "synthetic",
        "config": {"workload": workload, "sample": sample, "whole_config": whole},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": info["cores"], "kind": "port", "sample": sample,
                         "stages_s": info["stages_s"], "host_cpus": ncpu, "median_s": float(np.median(times)), "min_s": min(times)},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


DUMP_BYTES = 60_000_000  # the .npy files of --dump-outputs stay below 64 MB


def dump_outputs(d, pano, mask):
    """--dump-outputs: the panorama and mask of the last timed step, as float32 DIR/pano.npy (h x w x 3) and DIR/mask.npy
    (h x w).  When they would exceed DUMP_BYTES, a fixed sample of pixels (the same for the same panorama size) stands for them:
    DIR/pano_sample.npy (k x 3), DIR/mask_sample.npy (k) and their flat pixel indices DIR/pixel_index.npy (float64)."""
    os.makedirs(d, exist_ok=True)
    h, w = mask.shape
    per_pixel = 4 * 4  # float32 r, g, b, mask
    if h * w * per_pixel <= DUMP_BYTES:
        np.save(os.path.join(d, "pano.npy"), pano.astype(np.float32))
        np.save(os.path.join(d, "mask.npy"), mask.astype(np.float32))
        return
    idx = np.sort(np.random.default_rng(0).choice(h * w, DUMP_BYTES // (per_pixel + 8), replace=False))
    np.save(os.path.join(d, "pano_sample.npy"), pano.reshape(-1, 3)[idx].astype(np.float32))
    np.save(os.path.join(d, "mask_sample.npy"), mask.reshape(-1)[idx].astype(np.float32))
    np.save(os.path.join(d, "pixel_index.npy"), idx.astype(np.float64))


def set_extras(comp):
    """--extras: the other two FINAL-resolution steps of the pipeline fused into the step (SURVEY 8f f1, f2): a
    synthetic exposure gain map (one sample per 32x32 block, as gain_blocks estimates) and a LOW-resolution seam mask
    (keeps the middle three quarters of every image; the overlaps of the ring stay covered) per image."""
    rng = np.random.default_rng(5)
    for i, (_x, _y, w, h) in enumerate(comp.rects):
        comp.set_gain(i, rng.uniform(0.9, 1.1, (max(1, h // 32), max(1, w // 32))).astype(np.float32))
        sh, sw = max(2, int(round(h / 3.2))), max(2, int(round(w / 3.2)))
        seam = np.zeros((sh, sw), np.uint8)
        seam[:, sw // 8: sw - sw // 8] = 255
        comp.set_seam_mask(i, seam)


def dropin_e2e(cfg, imgs, reps=3):
    """The path the north_star names: the reference's own call sequence (stitcher.py:185-189, 219-225, 241-259) through the
    drop-in classes -- Warper.warp_images + create_and_warp_masks + warp_rois, Blender.prepare / feed / blend -- with host
    ndarrays in and out, every call synchronous like the reference's.  Returns (MPix/s, ms per composite, result)."""
    from stitching_b200 import Blender, Warper

    cams = cfg["cameras"]
    sizes = [(cfg["w"], cfg["h"])] * len(cams)
    times, stages = [], []
    pano = mask = None
    for _ in range(reps + 1):  # the first pass is the warm-up
        t = [time.perf_counter()]
        warper = Warper(cfg["warper"])
        warper.set_scale(cams)
        warped = list(warper.warp_images(imgs, cams))
        t.append(time.perf_counter())
        masks = list(warper.create_and_warp_masks(sizes, cams))
        t.append(time.perf_counter())
        corners, wsizes = warper.warp_rois(sizes, cams)
        blender = Blender(cfg["blender"], cfg["strength"])
        blender.prepare(corners, wsizes)
        t.append(time.perf_counter())
        for img, m, c in zip(warped, masks, corners):
            blender.feed(img, m, c)
        t.append(time.perf_counter())
        pano, mask = blender.blend()
        t.append(time.perf_counter())
        times.append(t[-1] - t[0])
        stages.append([b - a for a, b in zip(t, t[1:])])
    dt = float(np.median(times[1:]))
    mpix = len(cams) * cfg["w"] * cfg["h"] / 1e6
    names = ["warp_images", "create_and_warp_masks", "warp_rois+prepare", "feed", "blend"]
    stage_ms = {k: round(1e3 * float(np.median([st[i] for st in stages[1:]])), 2) for i, k in enumerate(names)}
    return mpix / dt, 1e3 * dt, pano, mask, stage_ms


def run_ours(args, rank, local_rank, world):
    from stitching_b200 import Compositor, _lib

    dist = Dist(world)
    L = _lib.lib()
    _lib.check(L.sb_init(local_rank), "sb_init")
    cfg, imgs = make_workload(args.workload, rank)
    n, w, h = cfg["n"], cfg["w"], cfg["h"]
    sizes = [(w, h)] * n
    t0 = time.perf_counter()
    comp = Compositor(cfg["cameras"], sizes, cfg["warper"], cfg["blender"], cfg["strength"])
    plan_ms = 1e3 * (time.perf_counter() - t0)
    mpix_rank = n * w * h / 1e6
    if args.extras:
        set_extras(comp)

    # ---- device-resident throughput (`value`) -----------------------------------------------------
    comp.upload(imgs)
    for _ in range(args.warmup):
        comp.run()
    comp.sync()
    # batches in flight: further compositors of the same rig (own stream, own buffers, own resident batch); the steps
    # are dealt round-robin so that the small latency-bound kernels of one step overlap the large ones of another
    from stitching_b200.compositor import time_multi

    extra = []
    for k in range(1, args.inflight):
        c2 = Compositor(cfg["cameras"], sizes, cfg["warper"], cfg["blender"], cfg["strength"])
        if args.extras:
            set_extras(c2)
        c2.upload(imgs)
        for _ in range(args.warmup):
            c2.run()
        c2.sync()
        extra.append(c2)
    single_ms, launches = comp.time(min(args.steps, 20), flush_l2=args.flush_l2)  # one batch at a time + per-kernel times
    single_ms /= min(args.steps, 20)
    dist.barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    launches0 = L.sb_launch_count()
    if extra:
        total_ms = time_multi([comp] + extra, args.steps)
    else:
        total_ms, launches = comp.time(args.steps, flush_l2=args.flush_l2)
    launches1 = L.sb_launch_count()
    comp.sync()
    for c2 in extra:
        c2.sync()
    clocks = sampler.result()
    if args.dump_outputs and rank == 0:  # the steps were dealt round-robin: the last one ran on this compositor
        dump_outputs(args.dump_outputs, *([comp] + extra)[(args.steps - 1) % (1 + len(extra))].download())
    dist.barrier()
    worst_ms = dist.max(total_ms)
    total_mpix = dist.sum(mpix_rank)
    ms_per_step = worst_ms / args.steps
    value = total_mpix / (ms_per_step * 1e-3)

    # ---- roofline of the dominant kernel ----------------------------------------------------------
    total_bytes, per_launch_bytes = comp.model_bytes()
    k_dom = int(np.argmax([ms for _, ms in launches]))
    dom_name, dom_ms = launches[k_dom]
    peak, peak_src = measured_peak_gbs()
    achieved = per_launch_bytes[k_dom] / (dom_ms * 1e-3) / 1e9
    roofline = {
        "bound": "hbm", "kernel": dom_name, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
        "traffic": ncu_traffic(dom_name), "peak_source": peak_src, "algorithmic_bytes": per_launch_bytes[k_dom],
        "kernel_ms": dom_ms,
        "whole_step": {"algorithmic_bytes": total_bytes, "achieved": total_bytes / (total_ms / args.steps * 1e-3) / 1e9,
                       "frac": total_bytes / (total_ms / args.steps * 1e-3) / 1e9 / peak},
        "launches_ms": {name: round(ms, 4) for name, ms in launches},
    }

    # ---- end to end through the public API with pinned host buffers (`e2e`) --------------------------
    src_bytes = h * w * 3
    _, _, pw, ph = comp.roi
    host_src = []
    for im in imgs:
        p = L.sb_host_alloc(src_bytes)
        if not p:
            _lib.check(-5, "sb_host_alloc")
        buf = np.ctypeslib.as_array((C.c_uint8 * src_bytes).from_address(p)).reshape(h, w, 3)
        buf[...] = im
        host_src.append((p, buf))
    p_pano, p_mask = L.sb_host_alloc(ph * pw * 3), L.sb_host_alloc(ph * pw)
    pano = np.ctypeslib.as_array((C.c_uint8 * (ph * pw * 3)).from_address(p_pano)).reshape(ph, pw, 3)
    pmask = np.ctypeslib.as_array((C.c_uint8 * (ph * pw)).from_address(p_mask)).reshape(ph, pw)

    def e2e_step():  # one step, nothing overlapped: latency of a single composite
        comp.upload([b for _, b in host_src], pinned=True)
        comp.run()
        comp.download(pano, pmask)  # synchronises

    for _ in range(3):
        e2e_step()
    dist.barrier()
    e2e_steps = max(4, min(args.steps, 40))
    t0 = time.perf_counter()
    for _ in range(3):
        e2e_step()
    latency_ms = 1e3 * (time.perf_counter() - t0) / 3
    # throughput: every step still uploads its inputs and downloads its result, but consecutive steps are
    # pipelined (two buffer sets, copy streams): sb_compositor_submit / sb_compositor_wait
    depth = 3  # buffer sets inside the compositor = results that may be in flight
    outs = [(pano, pmask)] + [(comp.pinned_empty((ph, pw, 3)), comp.pinned_empty((ph, pw))) for _ in range(depth - 1)]
    pano2 = outs[1][0]
    srcs = [b for _, b in host_src]
    for k in range(depth):
        comp.wait(comp.submit(srcs, *outs[k]))
    dist.barrier()
    t0 = time.perf_counter()
    tickets = []
    for k in range(e2e_steps):
        if k >= depth:
            comp.wait(tickets[k - depth])  # the host buffer of this slot has been delivered: it may be reused
        tickets.append(comp.submit(srcs, *outs[k % depth]))
    for t in tickets[-depth:]:
        comp.wait(t)
    e2e_s = dist.max(time.perf_counter() - t0)
    e2e = {"value": total_mpix * e2e_steps / e2e_s, "unit": UNIT, "h2d_bytes_per_step": n * src_bytes,
           "d2h_bytes_per_step": ph * pw * 4, "ms_per_step": 1e3 * e2e_s / e2e_steps, "steps": e2e_steps,
           "unpipelined_ms_per_step": latency_ms,
           "api": "stitching_b200.Compositor.submit/wait (sb_compositor_submit/_wait C ABI): per step H2D of the sources "
                  "from pinned host memory + warp/blend + D2H of panorama and mask; consecutive steps pipelined 3 deep"}
    assert np.array_equal(pano, pano2), "pipelined slots disagree"
    # the same step through the drop-in Warper / Blender classes (what stitcher.py calls), host ndarrays in and out
    dropin = None
    if rank == 0 and not args.no_dropin:
        dv, dms, dpano, dmask, dstages = dropin_e2e(cfg, imgs)
        dropin = {"value": dv, "unit": UNIT, "ms_per_step": dms, "stage_ms": dstages, "h2d_bytes_per_step": n * src_bytes, "d2h_bytes_per_step": ph * pw * 4,
                  "identical_to_compositor": bool(np.array_equal(dpano, pano) and np.array_equal(dmask, pmask)),
                  "api": "stitching_b200.Warper.warp_images / create_and_warp_masks / warp_rois + Blender.prepare / feed / blend "
                         "(the calls of stitcher.py:185-189, 241-259): pageable host ndarrays in and out, one synchronous call per image and stage"}
        e2e["dropin"] = dropin
    checksum = int(pano[::97, ::89].astype(np.uint64).sum())  # the result was really produced and read back

    # ---- CPU baseline: the reference's cv2 path on this box's host cores (rank 0, N = 1 only), and parity ------
    cpu, parity = None, None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu, parity = cpu_baseline_block(cfg, imgs, np.array(pano), np.array(pmask))

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "int16+f32 (uint8 in/out)", "data": "synthetic",
            "config": {
                "workload": f"{args.workload}: {WORKLOADS[args.workload]}" + (f" SCALED DOWN x{SCALE_DOWN} (debug)" if SCALE_DOWN != 1 else "") +
                            (" + fused exposure gains and seam masks (--extras; not the BASELINE metric's step)" if args.extras else ""),
                "images_per_gpu": n, "pano": [pw, ph],
                "num_bands": comp.num_bands, "plan_ms": round(plan_ms, 2),
                "batches_in_flight": args.inflight, "one_batch_at_a_time_ms_per_step": round(single_ms, 4),
                "l2": "L2 flushed between steps" if args.flush_l2 else
                      f"no flush: a step streams {total_bytes / 1e6:.0f} MB, inputs {n * src_bytes / 1e6:.0f} MB > 126 MB L2",
                "parallelism": "1 GPU" if world == 1 else f"{world} GPUs, one independent {n}-image ring per GPU (no collective)",
                "timed": "plan (roi detection, trig tables, buffers) built once outside the timed region; a step = warp + pyramids + collapse kernels",
                "source_layout": ("one word per pixel (r | g<<8 | b<<16): every upload is followed by a repack kernel on the copy stream, outside "
                                  "`value`'s timed region (inputs resident) and inside `e2e`'s; SB_SRC4=0 keeps the packed 3-byte sources"
                                  if os.environ.get("SB_SRC4", "1") != "0" else "packed 3-byte sources (SB_SRC4=0)"),
            },
            "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches1 - launches0), "roofline": roofline,
            "cpu_baseline": cpu, "parity": parity, "result_checksum": checksum,
        }
        print(json.dumps(line), flush=True)
    for p, _ in host_src:
        L.sb_host_free(p)
    L.sb_host_free(p_pano)
    L.sb_host_free(p_mask)
    for c2 in extra:
        c2.close()
    comp.close()
    dist.close()


def run_sharded(args, rank, local_rank, world):
    """N > 1: ONE panorama over N GPUs (BASELINE configs[2] family): 4 images of 4000x3000 per GPU on a cylindrical
    ring (f = 8000, 10 degree step; N = 8 is configs[2] itself), each rank warps + pyramids its block and the per-band
    partial sums where footprints cross strip boundaries travel over NVLink (NCCL send/recv), then every rank
    collapses its own column strip.  Weak scaling: per-GPU work is fixed."""
    from stitching_b200 import Compositor, _lib, rigs
    from stitching_b200 import dist as sbdist

    # NCCL's own log lines (NCCL_DEBUG=INFO from the driver) go to stderr unless the caller chose a file: stdout
    # carries the one JSON line
    if os.environ.get("NCCL_DEBUG") and not os.environ.get("NCCL_DEBUG_FILE"):
        os.environ["NCCL_DEBUG_FILE"] = "/dev/stderr"
    dist = Dist(world)
    L = _lib.lib()

    def bcast(payload):
        box = [payload]
        dist.pg.broadcast_object_list(box, src=0)
        return box[0]

    sbdist.init_comm(rank, world, bcast, device=local_rank)
    grid = args.workload == "cfg5"  # BASELINE configs[4]: the 16-image affine grid + feather, the SAME 16 images over N GPUs
    if grid:
        cfg = rigs.config("cfg5", SCALE_DOWN)
        n, w, h, cams, warper, blender = cfg["n"], cfg["w"], cfg["h"], cfg["cameras"], cfg["warper"], cfg["blender"]
        per_gpu = n // world
    else:
        per_gpu, w, h = 4, 4000 // SCALE_DOWN, 3000 // SCALE_DOWN
        n = per_gpu * world
        cams, warper, blender = rigs.yaw_ring(n, w, h, 8000 / SCALE_DOWN, 10), "cylindrical", "multiband"
    t0 = time.perf_counter()
    comp = Compositor(cams, [(w, h)] * n, warper, blender, 5, rank=rank, world=world)
    plan_ms = 1e3 * (time.perf_counter() - t0)
    imgs = [rigs.synth_image(h, w, i) for i in range(comp.first, comp.first + comp.count)]
    comp.upload(imgs)
    for _ in range(args.warmup):
        comp.run()
    comp.sync()
    dist.barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    launches0 = L.sb_launch_count()
    total_ms, launches = comp.time(args.steps)
    launches1 = L.sb_launch_count()
    comp.sync()
    clocks = sampler.result()
    dist.barrier()
    worst_ms = dist.max(total_ms)
    total_mpix = n * w * h / 1e6
    ms_per_step = worst_ms / args.steps
    value = total_mpix / (ms_per_step * 1e-3)
    slab_bytes = sum(comp.shard_slab(p, True)[1] for p in range(world) if p != rank)
    slab_total = dist.sum(slab_bytes)

    # end to end: every rank uploads its block from pinned host memory and reads its strip back, every step
    src_bytes = h * w * 3
    host = [comp.pinned_empty((h, w, 3)) for _ in imgs]
    for b, im in zip(host, imgs):
        b[...] = im
    sw = comp.strip[1] - comp.strip[0]  # columns of the panorama, or rows when the blocks are stacked (feather grid)
    rows = comp.strip_axis == 1
    ph, pw = (sw, comp.roi[2]) if rows else (comp.roi[3], sw)
    pano, pmask = comp.pinned_empty((max(ph, 1), max(pw, 1), 3)), comp.pinned_empty((max(ph, 1), max(pw, 1)))

    def e2e_step():
        comp.upload(host, pinned=True)
        comp.run()
        if sw > 0:
            comp.download(pano, pmask)  # synchronises
        else:
            comp.sync()

    for _ in range(3):
        e2e_step()
    dist.barrier()
    e2e_steps = max(4, min(args.steps, 40))
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step()
    dist.barrier()
    e2e_s = dist.max(time.perf_counter() - t0)
    h2d = dist.sum(len(imgs) * src_bytes)
    d2h = dist.sum(ph * pw * 4)

    # ---- parity of the sharded result (outside every timed region): every rank's strip against ONE single-GPU
    # composite of the whole ring computed on rank 0's GPU.  int16 sums are exact under any grouping; the float weight
    # sums are grouped per rank (re-associated where images of three or more ranks meet): +-1 LSB is the stated bar.
    import torch

    parity, like_for_like = None, None
    strips = [None] * world
    dist.pg.all_gather_object(strips, (int(comp.strip[0]), int(comp.strip[1])))
    if rank == 0:
        t0 = time.perf_counter()
        whole = Compositor(cams, [(w, h)] * n, warper, blender, 5)
        ref_pano, ref_mask = whole.composite([rigs.synth_image(h, w, i) for i in range(n)])
        whole_ms = None
        if grid:  # strong scaling: the N = 1 point is this very configuration on one GPU
            for _ in range(args.warmup):
                whole.run()
            whole.sync()
            whole_ms, _ = whole.time(args.steps)
        whole.close()
        differing, max_abs, mask_diff, values = 0, 0, 0, 0
        for r in range(world):
            lo, hi = strips[r]
            if hi <= lo:
                continue
            if r == 0:
                sp, sm = np.array(pano), np.array(pmask)
            else:
                shape = (hi - lo, comp.roi[2]) if rows else (comp.roi[3], hi - lo)
                tp = torch.empty(shape + (3,), dtype=torch.uint8)
                tm = torch.empty(shape, dtype=torch.uint8)
                dist.pg.recv(tp, src=r)
                dist.pg.recv(tm, src=r)
                sp, sm = tp.numpy(), tm.numpy()
            want, want_mask = (ref_pano[lo:hi], ref_mask[lo:hi]) if rows else (ref_pano[:, lo:hi], ref_mask[:, lo:hi])
            d = np.abs(sp.astype(np.int16) - want.astype(np.int16))
            differing += int(np.count_nonzero(d))
            max_abs = max(max_abs, int(d.max()) if d.size else 0)
            mask_diff += int(np.count_nonzero(sm != want_mask))
            values += int(sp.size)
        parity = {"differing": differing, "max_abs": max_abs, "mask_differing": mask_diff, "values": values,
                  "against": f"a single-GPU composite of the same {n} images on rank 0 (strips gathered over gloo), {time.perf_counter() - t0:.1f} s"}
        if grid:
            like_for_like = {"value": total_mpix / (whole_ms / args.steps * 1e-3), "unit": UNIT, "ms_per_step": whole_ms / args.steps,
                             "workload": f"the same {n}x{w}x{h} affine + feather configuration on ONE GPU (strong scaling: total work fixed)"}
        else:
            # like-for-like weak-scaling baseline: ONE GPU compositing 4 images of the same ring (the per-GPU work of this run)
            one = Compositor(cams[:per_gpu], [(w, h)] * per_gpu, warper, blender, 5)
            one.upload([rigs.synth_image(h, w, i) for i in range(per_gpu)])
            for _ in range(args.warmup):
                one.run()
            one.sync()
            one_ms, _ = one.time(args.steps)
            one.close()
            like_for_like = {"value": per_gpu * w * h / 1e6 / (one_ms / args.steps * 1e-3), "unit": UNIT, "ms_per_step": one_ms / args.steps,
                             "workload": f"{per_gpu}x{w}x{h} cylindrical + multiband on ONE GPU: the first {per_gpu} images of the same ring "
                                         f"(the N = 1 point of this weak-scaling family; `bench.py --gpus 1` runs BASELINE configs[1] instead)"}
    elif sw > 0:
        dist.pg.send(torch.from_numpy(np.ascontiguousarray(pano)), dst=0)
        dist.pg.send(torch.from_numpy(np.ascontiguousarray(pmask)), dst=0)
    dist.barrier()
    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong" if grid else "weak", "vs_baseline": None,
            "dtype": "int16+f32 (uint8 in/out)", "data": "synthetic",
            "config": {
                "workload": (f"cfg5: {n}x{w}x{h} RGB, affine plane warp + feather blend over {world} GPUs (BASELINE configs[4])" if grid
                             else sharded_workload_name(n, w, h, world)),
                "strips": "rows" if rows else "columns",
                "images_per_gpu": per_gpu, "pano": [comp.roi[2], comp.roi[3]], "num_bands": comp.num_bands, "plan_ms": round(plan_ms, 2),
                "parallelism": f"{world} GPUs: image blocks per rank, pano {'row' if rows else 'column'} strips per rank; the partial sums that cross strip "
                               f"boundaries go to the owner's memory over NVLink (copy engine + flags; SB_PEER=0: grouped NCCL send/recv) on a "
                               f"communication stream, overlapped with the kernels ({slab_total / 1e6:.1f} MB per step in total)",
                "l2": f"no flush: each rank streams its {per_gpu * src_bytes / 1e6:.0f} MB of sources every step (> 126 MB L2)",
                "timed": ("plan built once; a step = warp + distance-transform weights + partial sums + exchange + normalise of the own strip" if grid else
                          "plan built once; a step = warp + pyramids + partial sums + exchange (level-0 slabs leave after the first pyrDown) + collapse of the own strip"),
                "like_for_like_n1": like_for_like,
            },
            "clocks": clocks,
            "e2e": {"value": total_mpix * e2e_steps / e2e_s, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "ms_per_step": 1e3 * e2e_s / e2e_steps, "steps": e2e_steps,
                    "api": "stitching_b200.Compositor(rank, world).upload/run/download per rank, pinned host buffers"},
            "gpu_launches": int(launches1 - launches0),
            "roofline": {"bound": "hbm", "kernel": None, "achieved": None, "peak": measured_peak_gbs()[0], "unit": "GB/s", "frac": None,
                         "traffic": None, "note": "per-kernel roofline is reported at N = 1", "launches_ms_rank0": {k: round(v, 4) for k, v in launches}},
            "cpu_baseline": None, "parity": parity,
            "result_checksum": int(pano[::97, ::89].astype(np.uint64).sum()),
        }
        print(json.dumps(line), flush=True)
    comp.close()
    sbdist.shutdown()
    dist.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--workload", choices=sorted(WORKLOADS), default="cfg2")
    ap.add_argument("--flush-l2", action="store_true")
    ap.add_argument("--inflight", type=int, default=2, help="N = 1: independent batches in flight (own stream + buffers each)")
    ap.add_argument("--cpu-sample", type=int, default=0, help="images of the ring per step of the reference arm (default: the whole configuration)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-dropin", action="store_true", help="skip the end-to-end measurement through the drop-in Warper / Blender classes")
    ap.add_argument("--replicas", action="store_true", help="N > 1: one independent panorama per GPU instead of one sharded panorama")
    ap.add_argument("--extras", action="store_true", help="also fuse exposure gains and seam masks into the step (SURVEY 8f f1, f2)")
    ap.add_argument("--scale-down", type=int, default=1, help="debug: shrink the workload (not a valid measurement)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the panorama and mask of the last timed step (rank 0) as .npy files to DIR; "
                                                          "--impl ours on one GPU or with --replicas only (not the sharded or reference paths)")
    args = ap.parse_args()
    global SCALE_DOWN
    SCALE_DOWN = args.scale_down
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    rank, local_rank, world = dist_env()
    if args.dump_outputs and (args.impl == "reference" or (world > 1 and not args.replicas)):
        ap.error("--dump-outputs: only the single-panorama path (--impl ours on one GPU, or --replicas)")
    if args.impl == "reference":
        run_reference(args, rank, world)
    elif world > 1 and not args.replicas:
        run_sharded(args, rank, local_rank, world)
    else:
        run_ours(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
