#!/usr/bin/env python
"""Times a zoom batch (fs_render_perturb_lav2_frames) against the same frames rendered one call at a time, on View 14
at 3840x2160, GpuHDRx32PerturbedLAv2: K frames at scales 2^(j/8), j = 0 .. K-1, sharing View 14's orbit and LA table.

    python tools/zoom_time.py [--frames 16] [--gpus 1,2,4,8] [--steps K] [--warmup W] [--out FILE]

One renderer (fs_create) and device groups of the listed sizes: on the machine's separate GPUs where it has enough of
them, else that many members sharing GPU 0 (the line says which).  Per configuration (one JSON line each):
* batch_ms       ClearMemory, then one batch call, ending in a synchronise of the compute streams: host clock, mean of K
* batch_device_ms  fs_last_render_ms of the batch (one launch; a group's slowest member)
* singles_ms     the same frames enqueued back to back as single renders, ending in a synchronise: host clock, mean of K
* frames_per_s_batch / frames_per_s_singles   frames / the two times
The two forms alternate step by step in the same process; the L2 is overwritten (256 MB) before every timed window.
Every frame's Min/Max/Sum after SelectFrame(k) is checked against a single render of that frame before any timing.
The card's name and power limit (nvidia-smi) are read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=16)
    ap.add_argument("--gpus", default="1,2,4,8", help="group sizes timed after the single renderer")
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
        raise SystemExit("zoom_time.py: no CUDA device")
    n_dev = torch.cuda.device_count()
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip().splitlines()

    alg = RenderAlgorithm.GpuHDRx32PerturbedLAv2
    w, h, K = args.width, args.height, args.frames
    p = PRESETS[14]
    view = View(p.min_x, p.min_y, p.max_x, p.max_y, w, h)
    numeric = traits(alg).numeric
    scales = [f"{2 ** (j / 8):.17g}" for j in range(K)]
    frames = [view.zoomed(s).coords(numeric) for s in scales]
    orbit = Orbit(view, numeric, p.num_iterations, True)
    la = LaTable(orbit, 4)
    n_iter = p.num_iterations

    configs = [("renderer", None)]
    for n in (int(x) for x in args.gpus.split(",")):
        configs.append((f"group{n}", list(range(n)) if n <= n_dev else [0] * n))

    lines = []
    for name, devices in configs:
        used = sorted(set(devices or [0]))
        flush = [torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=f"cuda:{d}") for d in used]  # > 126 MB L2
        r = GPURenderer(0) if devices is None else GPURenderer(devices=devices)
        assert r.InitializeMemory(w, h, 1, iter_bytes=4) == 0
        assert r.InitializePerturb(1, orbit, 0, None, la) == 0

        # the batch's frames against single renders of the same coordinates
        r.ClearMemory()
        want = []
        for c in frames:
            assert r.RenderPerturbLAv2(alg, c, n_iter) == 0
            rc, _, _, red = r.RenderCurrent(n_iter, want_iters=False)
            assert rc == 0
            want.append(red)
        r.ClearMemory()
        assert r.RenderPerturbLAv2Frames(alg, frames, n_iter) == 0
        for k in range(K):
            assert r.SelectFrame(k) == 0
            rc, _, _, red = r.RenderCurrent(n_iter, want_iters=False)
            assert rc == 0 and red == want[k], (name, k, red, want[k])

        def settle():
            for f in flush:
                f.zero_()
            for d in used:
                torch.cuda.synchronize(d)
            r.ClearMemory()
            assert r.SyncComputeStream() == 0

        def batch():
            settle()
            t0 = time.perf_counter()
            assert r.RenderPerturbLAv2Frames(alg, frames, n_iter) == 0
            assert r.SyncComputeStream() == 0
            return (time.perf_counter() - t0) * 1e3, r.LastRenderMs()

        def singles():
            settle()
            t0 = time.perf_counter()
            for c in frames:
                assert r.RenderPerturbLAv2(alg, c, n_iter) == 0
            assert r.SyncComputeStream() == 0
            return (time.perf_counter() - t0) * 1e3

        for _ in range(args.warmup):
            batch()
            singles()
        b, s = [], []
        for i in range(args.steps):
            if i % 2:
                s.append(singles())
                b.append(batch())
            else:
                b.append(batch())
                s.append(singles())
        r.close()
        del flush
        batch_ms = sum(x for x, _ in b) / len(b)
        singles_ms = sum(s) / len(s)
        line = {"config": name, "devices": devices if devices is not None else [0],
                "separate_gpus": devices is None or len(set(devices)) == len(devices),
                "workload": f"view14 GpuHDRx32PerturbedLAv2 {w}x{h} u32, {K} frames at 2^(j/8)",
                "batch_ms": batch_ms, "batch_ms_min": min(x for x, _ in b), "batch_ms_max": max(x for x, _ in b),
                "batch_device_ms": sum(d for _, d in b) / len(b),
                "singles_ms": singles_ms, "singles_ms_min": min(s), "singles_ms_max": max(s),
                "frames_per_s_batch": K / batch_ms * 1e3, "frames_per_s_singles": K / singles_ms * 1e3,
                "speedup": singles_ms / batch_ms, "frame_sums": [x["Sum"] for x in want],
                "steps": args.steps, "card": card}
        print(json.dumps(line), flush=True)
        lines.append(line)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(lines, f, indent=1)


if __name__ == "__main__":
    main()
