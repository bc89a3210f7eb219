#!/usr/bin/env python
"""Times one device group (fs_create_group) per GPU count on View 14, 3840x2160, GpuHDRx32PerturbedLAv2: the
single-process counterpart of `torchrun --nproc_per_node N bench.py --gpus N`.

    python tools/group_time.py [--gpus 1,2,4,8] [--steps K] [--warmup W] [--out FILE]
    python tools/group_time.py --devices "0;0,0;0,0,0,0"   # explicit groups (ids may repeat: shards sharing one GPU)

Per GPU count (one JSON line each):
* device_ms     ClearMemory + render, L2 overwritten before every step; fs_last_render_ms (slowest member), mean of K
* enqueue_ms    host time of the render call: one thread enqueues on every member
* e2e_sink_ms   InitializePerturb (page-locked tables) -> ClearMemory -> render -> RenderCurrent into a page-locked frame
                the members stream into while they render (result sink), wall clock per step
* e2e_copy_ms   the same without the sink: every member copies its bands after its render
* aa1_colour_ms / aa3_colour_ms  the same step on the 1280x720 colour frame of a 3840x2160 render at AA 3 (colours
                and Min/Max/Sum on the lead, after the members' bands crossed to it), and at AA 1 with colours (every
                member colours its own bands): the two sides of the result path's antialiasing choice
Every line carries the frame's Sum, which must be the same at every GPU count.
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
    ap.add_argument("--gpus", default="1,2,4,8")
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--devices", default=None, help="semicolon-separated device lists; replaces --gpus")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import numpy as np
    import torch
    from fractalshark_b200 import RenderAlgorithm, traits
    from fractalshark_b200.gpu_renderer import GPURenderer
    from fractalshark_b200.host_inputs import LaTable, Orbit, ReplicatedInputs, View
    from fractalshark_b200.views import PRESETS

    if not torch.cuda.is_available() or not GPURenderer.TestCudaIsWorking():
        raise SystemExit("group_time.py: no CUDA device")
    n_dev = torch.cuda.device_count()
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip().splitlines()

    alg = RenderAlgorithm.GpuHDRx32PerturbedLAv2
    w, h = 3840, 2160
    p = PRESETS[14]
    view = View(p.min_x, p.min_y, p.max_x, p.max_y, w, h)
    numeric = traits(alg).numeric
    coords = view.coords(numeric)
    orbit = Orbit(view, numeric, p.num_iterations, True)
    la = LaTable(orbit, 4)
    n_iter = p.num_iterations
    meta, blobs = ReplicatedInputs.pack(coords, orbit, la, n_iter)
    pinned = []
    for b in blobs:
        t = torch.empty(max(int(b.size), 1), dtype=torch.uint8, pin_memory=True)
        t[:b.size] = torch.from_numpy(b)
        pinned.append(t.numpy()[:b.size])
    _, orbit_pinned, la_pinned, _ = ReplicatedInputs.unpack(meta, pinned)

    def pinned_frame(shape, dtype=np.uint32):
        n = int(np.prod(shape)) * np.dtype(dtype).itemsize
        return torch.empty(n, dtype=torch.uint8, pin_memory=True).numpy().view(dtype).reshape(shape)

    lines = []
    if args.devices:
        groups = [[int(x) for x in g.split(",")] for g in args.devices.split(";")]
    else:
        groups = [list(range(int(n))) for n in args.gpus.split(",")]
    for devices in groups:
        n = len(devices)
        if max(devices) >= n_dev:
            print(json.dumps({"devices": devices, "skipped": f"{n_dev} devices"}), flush=True)
            continue
        flush = [torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=f"cuda:{d}") for d in sorted(set(devices))]  # > 126 MB L2
        r = GPURenderer(devices=devices)
        assert r.DeviceCount() == n
        assert r.InitializeMemory(w, h, 1, iter_bytes=4) == 0
        gen = 1
        assert r.InitializePerturb(gen, orbit, 0, None, la) == 0
        hp, wp = r.buffer_shape()

        def step_device():
            for f in flush:
                f.zero_()
            torch.cuda.synchronize()   # current device; the others are synchronised below
            for d in set(devices):
                torch.cuda.synchronize(d)
            r.ClearMemory()
            t0 = time.perf_counter()
            assert r.RenderPerturbLAv2(alg, coords, n_iter) == 0
            enq = (time.perf_counter() - t0) * 1e3
            assert r.SyncComputeStream() == 0
            return r.LastRenderMs(), enq

        for _ in range(args.warmup):
            step_device()
        dev = [step_device() for _ in range(args.steps)]
        rc, iters, _, red = r.RenderCurrent(n_iter)
        assert rc == 0
        frame_sum = red["Sum"]
        assert frame_sum == int(iters[:h, :w].astype(np.uint64).sum())

        frame = pinned_frame((hp, wp))

        def step_e2e(colours=False):
            nonlocal gen
            gen += 1
            assert r.InitializePerturb(gen, orbit_pinned, 0, None, la_pinned) == 0
            r.ClearMemory()
            assert r.RenderPerturbLAv2(alg, coords, n_iter) == 0
            rc, _, _, rd = r.RenderCurrent(n_iter, iters_out=frame, want_colors=colours)
            assert rc == 0 and rd["Sum"] == frame_sum
            return rd

        def timed(fn):
            for _ in range(2):
                fn()
            t0 = time.perf_counter()
            for _ in range(args.steps):
                fn()
            return (time.perf_counter() - t0) * 1e3 / args.steps

        e2e_copy = timed(step_e2e)
        assert r.SetResultSink(frame) == 0
        e2e_sink = timed(step_e2e)
        assert int(frame[:h, :w].astype(np.uint64).sum()) == frame_sum
        assert r.SetResultSink(None) == 0
        aa1 = timed(lambda: step_e2e(True))
        assert r.InitializeMemory(w, h, 3, iter_bytes=4) == 0
        aa3 = timed(lambda: step_e2e(True))
        r.close()
        del flush
        ms = [d for d, _ in dev]
        line = {"gpus": n, "devices": devices, "workload": "view14 GpuHDRx32PerturbedLAv2 3840x2160 u32",
                "device_ms": sum(ms) / len(ms), "device_ms_min": min(ms), "device_ms_max": max(ms),
                "enqueue_ms": sum(e for _, e in dev) / len(dev),
                "e2e_sink_ms": e2e_sink, "e2e_copy_ms": e2e_copy, "aa1_colour_ms": aa1, "aa3_colour_ms": aa3,
                "sum": frame_sum, "steps": args.steps, "card": card}
        print(json.dumps(line), flush=True)
        lines.append(line)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(lines, f, indent=1)


if __name__ == "__main__":
    main()
