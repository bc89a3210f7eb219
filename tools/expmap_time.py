#!/usr/bin/env python
"""Times an exponential map (fs_render_perturb_lav2_expmap) against the zoom batch of tools/zoom_time.py on View 14,
GpuHDRx32PerturbedLAv2, u32 counts, one renderer each, in the same process:

* the batch: K frames at 3840x2160, scales 2^(j/8), j = 0 .. K-1 (fs_render_perturb_lav2_frames, one launch);
* the exp map: W = 3840 columns around the same centre, from the largest frame's corners inwards down to the deepest
  frame's pixel spacing: rows = ceil(W ln Z / (2 pi)), Z = 2^((K-1)/8) * (half-diagonal of a frame in pixels).  For
  K = 16 that is 5,499 rows (21.1 M cells against the batch's 132.7 M).

    python tools/expmap_time.py [--frames 16] [--steps K] [--warmup W] [--out FILE]

Per form: ClearMemory, one render call ending in a synchronise of the compute stream (host clock, mean / min / max of
K steps) and fs_last_render_ms (device); cells/s = rendered cells / host time; Min/Max/Sum of the map and of every
frame.  The two forms alternate step by step and the L2 is overwritten (256 MB) before every timed window.  The card's
name and power limit (nvidia-smi) are read in the same run.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=16)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--width", type=int, default=3840)
    ap.add_argument("--height", type=int, default=2160)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    from fractalshark_b200 import RenderAlgorithm, traits
    from fractalshark_b200.gpu_renderer import GPURenderer
    from fractalshark_b200.host_inputs import LaTable, Orbit, View
    from fractalshark_b200.views import PRESETS

    if not torch.cuda.is_available() or not GPURenderer.TestCudaIsWorking():
        raise SystemExit("expmap_time.py: no CUDA device")
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip().splitlines()

    alg = RenderAlgorithm.GpuHDRx32PerturbedLAv2
    w, h, K = args.width, args.height, args.frames
    p = PRESETS[14]
    view = View(p.min_x, p.min_y, p.max_x, p.max_y, w, h)
    numeric = traits(alg).numeric
    scales = [f"{2 ** (j / 8):.17g}" for j in range(K)]
    frames = [view.zoomed(s).coords(numeric) for s in scales]
    zoom = 2 ** ((K - 1) / 8) * math.hypot(w, h) / 2
    rows = math.ceil(w * math.log(zoom) / (2 * math.pi))
    expmap = view.zoomed(scales[-1]).exp_map(numeric, rows)
    orbit = Orbit(view, numeric, p.num_iterations, True)
    la = LaTable(orbit, 4)
    n_iter = p.num_iterations

    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda:0")  # > 126 MB L2
    rb, rm = GPURenderer(0), GPURenderer(0)
    assert rb.InitializeMemory(w, h, 1, iter_bytes=4) == 0
    assert rm.InitializeMemory(w, rows, 1, iter_bytes=4) == 0
    for r in (rb, rm):
        assert r.InitializePerturb(1, orbit, 0, None, la) == 0

    def settle(r):
        flush.zero_()
        torch.cuda.synchronize(0)
        r.ClearMemory()
        assert r.SyncComputeStream() == 0

    def batch():
        settle(rb)
        t0 = time.perf_counter()
        assert rb.RenderPerturbLAv2Frames(alg, frames, n_iter) == 0
        assert rb.SyncComputeStream() == 0
        return (time.perf_counter() - t0) * 1e3, rb.LastRenderMs()

    def exp_map():
        settle(rm)
        t0 = time.perf_counter()
        rc = rm.RenderPerturbLAv2ExpMap(alg, expmap, n_iter)
        assert rc == 0, GPURenderer.ConvertErrorToString(rc)
        assert rm.SyncComputeStream() == 0
        return (time.perf_counter() - t0) * 1e3, rm.LastRenderMs()

    for _ in range(args.warmup):
        batch()
        exp_map()
    b, m = [], []
    for i in range(args.steps):
        if i % 2:
            m.append(exp_map())
            b.append(batch())
        else:
            b.append(batch())
            m.append(exp_map())

    frame_red = []
    for k in range(K):
        assert rb.SelectFrame(k) == 0
        rc, _, _, red = rb.RenderCurrent(n_iter, want_iters=False)
        assert rc == 0
        frame_red.append(red)
    rc, _, _, map_red = rm.RenderCurrent(n_iter, want_iters=False)
    assert rc == 0
    rb.close()
    rm.close()

    def stats(xs, cells):
        host = [x for x, _ in xs]
        mean = sum(host) / len(host)
        return {"ms": mean, "ms_min": min(host), "ms_max": max(host), "device_ms": sum(d for _, d in xs) / len(xs),
                "cells": cells, "cells_per_s": cells / mean * 1e3}

    line = {"workload": f"view14 GpuHDRx32PerturbedLAv2 u32; exp map {w}x{rows} vs {K} frames {w}x{h} at 2^(j/8)",
            "zoom_factor": zoom, "rows": rows, "log2_radius0": expmap["log2_radius0"],
            "log2_row_step": expmap["log2_row_step"],
            "expmap": dict(stats(m, w * rows), reduction=map_red),
            "batch": dict(stats(b, w * h * K), frame_reductions=frame_red),
            "steps": args.steps, "warmup": args.warmup, "l2": "overwritten (256 MB) before every timed window",
            "card": card}
    print(json.dumps(line), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(line, f, indent=1)


if __name__ == "__main__":
    main()
