"""End-to-end throughput of the pipelined Compositor.submit / wait path with BGR and YUV 4:2:0 frames (one B200).

Arms (all in one process, alternating round by round, pinned host buffers, the same number of steps each):
  bgr->bgr+mask     what bench.py's `e2e` measures
  nv12->bgr+mask    NV12 sources (half the upload bytes), BGR panorama and mask
  nv12->nv12        NV12 sources and NV12 panorama, no mask
  i420->i420        the same with I420
Prints one JSON line: per arm MPix/s of source pixels and ms per step (median over rounds, and every round), bytes up and
down per step, and a parity block -- differing values of the last step's outputs against the BGR composite of the
oracle-converted frames (tests/yuv_oracle.py), converted back by the oracle for YUV output.  The card's name and power
limit are read in the same run.

    python profiles/yuv_e2e.py [--workload cfg2|cfg3|cfg4] [--steps 40] [--rounds 5]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import yuv_oracle as YO  # noqa: E402
from stitching_b200 import Compositor, _lib, color, rigs  # noqa: E402

ARMS = [("bgr", "bgr", True), ("nv12", "bgr", True), ("nv12", "nv12", False), ("i420", "i420", False)]
DEPTH = 3


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = (s.strip() for s in out.split(","))
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:  # the numbers are still printed, without the card's description
        return {"error": str(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="cfg2", choices=["cfg2", "cfg3", "cfg4"])
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--rounds", type=int, default=5)
    args = ap.parse_args()
    _lib.check(_lib.lib().sb_init(0), "sb_init")
    cfg = rigs.config(args.workload, 1)
    n, w, h = cfg["n"], cfg["w"], cfg["h"]
    comp = Compositor(cfg["cameras"], [(w, h)] * n, cfg["warper"], cfg["blender"], cfg["strength"])
    _, _, pw, ph = comp.roi
    bgr = [rigs.synth_image(h, w, i) for i in range(n)]
    inputs = {"bgr": bgr}
    for fmt in ("nv12", "i420"):
        inputs[fmt] = [YO.bgr_to_yuv420(im, fmt) for im in bgr]
    pinned = {}
    for fmt, frames in inputs.items():
        pinned[fmt] = [comp.pinned_empty(f.shape) for f in frames]
        for p, f in zip(pinned[fmt], frames):
            p[...] = f
    outs = {}
    for fi, fo, with_mask in ARMS:
        outs[(fi, fo)] = [(comp.pinned_empty(color.frame_shape(pw, ph, fo)), comp.pinned_empty((ph, pw)) if with_mask else None)
                          for _ in range(DEPTH)]

    def run(fi, fo, steps):
        o = outs[(fi, fo)]
        tickets = []
        t0 = time.perf_counter()
        for k in range(steps):
            if k >= DEPTH:
                comp.wait(tickets[k - DEPTH])
            tickets.append(comp.submit(pinned[fi], o[k % DEPTH][0], o[k % DEPTH][1], in_fmt=fi, out_fmt=fo))
        for t in tickets[-DEPTH:]:
            comp.wait(t)
        return time.perf_counter() - t0, (steps - 1) % DEPTH

    for fi, fo, _ in ARMS:  # warm-up: every slot of every arm (graph capture, first-use allocations)
        run(fi, fo, 2 * DEPTH)
    times = {(fi, fo): [] for fi, fo, _ in ARMS}
    last = {}
    for _ in range(args.rounds):
        for fi, fo, _m in ARMS:
            s, slot = run(fi, fo, args.steps)
            times[(fi, fo)].append(1e3 * s / args.steps)
            last[(fi, fo)] = slot

    # parity of the last step of every arm
    ref_bgr = {}
    for fmt in ("bgr", "nv12", "i420"):
        frames = inputs[fmt] if fmt == "bgr" else [YO.yuv420_to_bgr(f, fmt) for f in inputs[fmt]]
        ref_bgr[fmt] = tuple(a.copy() for a in comp.composite(frames))
    mpix = n * w * h / 1e6
    arms = {}
    for fi, fo, with_mask in ARMS:
        pano, mask = outs[(fi, fo)][last[(fi, fo)]]
        rp, rm = ref_bgr[fi]
        exp = rp if fo == "bgr" else YO.bgr_to_yuv420(rp, fo)
        up = n * (w * h * 3 if fi == "bgr" else w * h * 3 // 2)
        down = (pw * ph * 3 if fo == "bgr" else pw * ph * 3 // 2) + (pw * ph if with_mask else 0)
        ms = statistics.median(times[(fi, fo)])
        arms[f"{fi}->{fo}" + ("+mask" if with_mask else "")] = {
            "value": mpix / (ms * 1e-3), "unit": "MPix/s", "ms_per_step": ms, "ms_per_step_rounds": [round(t, 4) for t in times[(fi, fo)]],
            "h2d_bytes_per_step": up, "d2h_bytes_per_step": down,
            "parity": {"reference": "BGR composite of the oracle-converted frames" + (", oracle-converted to " + fo if fo != "bgr" else ""),
                       "differing_values": int((pano != exp).sum()), "values": int(exp.size),
                       "mask_differing_values": int((mask != rm).sum()) if with_mask else None},
        }
    line = {"metric": "yuv_e2e", "workload": args.workload, "images": n, "frame": [w, h], "pano": [pw, ph], "num_bands": comp.num_bands,
            "steps_per_round": args.steps, "rounds": args.rounds, "pipeline_depth": DEPTH, "card": card(),
            "timed": "host clock around `steps` pipelined submit/wait steps with pinned host buffers (every step uploads all sources "
                     "and downloads the panorama), arms alternating round by round; value = source MPix per second",
            "arms": arms}
    print(json.dumps(line), flush=True)
    comp.close()


if __name__ == "__main__":
    main()
