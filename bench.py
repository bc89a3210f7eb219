#!/usr/bin/env python
"""bench.py -- headline benchmark of the per-pixel render path (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # our arm (libfsgpu.so on N B200s)
    python bench.py --impl reference --gpus N --steps K ...  # reference arm: the reference's CPU renderer on host cores
    python bench.py --workload NAME                          # another BASELINE config as the headline (see WORKLOADS)
    python bench.py --dump-outputs DIR ...                   # also write the last timed step's frame to DIR/*.npy

Headline workload (config.workload): View #14 (north_star's target view: 6,632-digit coordinates, zoom 4.7e6516,
maxIter 2,147,483,646), GpuHDRx32PerturbedLAv2, 3840x2160, AA 1, u32 iterations (BASELINE.json configs[3]).  The
reference orbit comes from the in-tree GMP loop (21.7 kbit, period 116,695, a few seconds; untimed), the LA table from the
in-tree builder (byte-identical to the reference's LAReference.cpp: tests/test_table_construction.py).  One step =
ClearMemory + one full render of the frame.

* value        pixel-iterations/s = ReductionResults.Sum / device time of the render kernel(s), inputs (orbit, LA table)
               already resident in HBM; CUDA events on the launching stream, max over ranks.
* e2e          same metric through the public C-ABI call sequence with HOST buffers inside the timed region:
               InitializePerturb (H2D orbit + LA table), ClearMemory, RenderPerturbLAv2, RenderCurrent (AA/palette/
               reduction + the iteration buffer and the 24-byte reduction on the host).  Two variants on the line: `e2e`
               (page-locked inputs, frame streamed by the kernel into a page-locked sink) and `e2e_as_is` (pageable
               inputs and frame, exactly what an unmodified caller hands over).
* roofline     FP32 issue: EXECUTED FP32-pipe thread-instructions (steps by kind from device counters x the FP32
               instructions this kernel issues per step) / kernel time, against the FFMA issue peak measured live by a
               micro-kernel on the same GPU.  The reference formulation's work per step (SURVEY.md 8d) is reported
               separately as `reference_work_credit`.
* configs      the other BASELINE configs, one entry each: device time, the reference CUDA kernel beside it on the same
               GPU and inputs (oracle/_ref, the checker), pixels exact, roofline.
* cpu_baseline the reference's own CPU renderer (Fractal::CalcCpuPerturbationFractalLAV2, oracle/_ref/libref_host.so)
               on a bounded pixel sample with all host threads; the oracle's CPU port of the GPU algorithm beside it.
N > 1: 4-row tile bands are dealt round-robin to ranks (no data-path collective inside the render); the orbit/LA blob is
replicated by an NCCL broadcast.  The device-timed arm checks the merged frame with an NCCL reduce (disjoint rows, so
SUM == gather; untimed).  The e2e arm assembles the frame on the HOST: one shared-memory frame, page-locked by every rank.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

# ---- workloads: BASELINE.json configs as concrete inputs (BASELINE.md section 3) ------------------------------------
# kind: which render entry; n_iter None = the preset's limit; window = explicit bounds instead of a view preset.
WORKLOADS = {
    # configs[3]: the headline and its 2x32 sibling, plus View 19
    "view14_hdr32_lav2": dict(config=3, view=14, alg="GpuHDRx32PerturbedLAv2", w=3840, h=2160),
    "view14_hdr2x32_lav2": dict(config=3, view=14, alg="GpuHDRx2x32PerturbedLAv2", w=3840, h=2160),
    "view19_hdr32_lav2": dict(config=3, view=19, alg="GpuHDRx32PerturbedLAv2", w=3840, h=2160),
    "view14_hdr32_bla": dict(config=3, view=14, alg="GpuHDRx32PerturbedBLA", w=3840, h=2160),
    # configs[2]: View 5, BLA and LAv2 (+ perturbation only, capped: every counted iteration is an executed step)
    "view5_hdr32_bla": dict(config=2, view=5, alg="GpuHDRx32PerturbedBLA", w=3840, h=2160),
    "view5_hdr32_lav2": dict(config=2, view=5, alg="GpuHDRx32PerturbedLAv2", w=3840, h=2160),
    "view5_hdr32_lav2_po": dict(config=2, view=5, alg="GpuHDRx32PerturbedLAv2PO", w=3840, h=2160, n_iter=50000),
    # configs[1]: direct escape time, View 0 and an all-interior window (centre (-0.1, 0), 0.25 wide)
    "view0_f32_direct": dict(config=1, view=0, alg="Gpu1x32", w=3840, h=2160, n_iter=65536),
    "view0_f64_direct": dict(config=1, view=0, alg="Gpu1x64", w=3840, h=2160, n_iter=65536),
    "interior_f32_direct": dict(config=1, window=("-0.225", "-0.0703125", "0.025", "0.0703125"), alg="Gpu1x32", w=3840, h=2160,
                                n_iter=65536),
    "interior_f64_direct": dict(config=1, window=("-0.225", "-0.0703125", "0.025", "0.0703125"), alg="Gpu1x64", w=3840, h=2160,
                                n_iter=65536),
    # configs[4] stand-in: View 30's resolution and iteration limit on View 14's coordinates (north_star: "synthetic views
    # of the named resolution and iteration limit"; View 30's own 16384-limb orbit needs the reference's NTT producer)
    "view30_standin_8k": dict(config=4, view=14, alg="GpuHDRx32PerturbedLAv2", w=7680, h=4320, n_iter=200_000_000),
}
HEADLINE = "view14_hdr32_lav2"
DEFAULT_CONFIGS = ["view14_hdr2x32_lav2", "view19_hdr32_lav2", "view14_hdr32_bla", "view5_hdr32_bla", "view5_hdr32_lav2", "view5_hdr32_lav2_po",
                   "view0_f32_direct", "view0_f64_direct", "interior_f32_direct", "interior_f64_direct", "view30_standin_8k"]

# FP32-pipe thread-instructions the HDRx32 LAv2 kernel ISSUES per step (fs_lav2.cuh / fs_scaled_loop.cuh):
#   AT pass   FMUL2 (2) + FMUL + FADD + FFMA2 (2) = 6, plus one FADD per 16-pass chunk for the escape test
#   LA step   3 aligned complex additions (2 FFMA each) + 3 complex products (2 FMUL + 2 FFMA each) + Reduce (2 FMUL) + 2 scalings = 22
#             (the select-free alignment of fs_la_step2.cuh scales both operands and its range guards add three FADDs: 30 issued;
#             only the 22 are counted)
#   perturbation step (scaled plain-float chunk)  2 FFMA + 4 FMUL + 4 FADD + 1 FMUL of the threshold test = 11
EXECUTED_FP32 = {"at": 6.0 + 1.0 / 16.0, "la": 22.0, "perturbation": 11.0}
# work per step of the reference formulation (SURVEY.md section 8d; AT pass: rr, ii, rr+ii, rr-ii, re*im, 3 FMA + compare)
REFERENCE_CREDIT = {"at": 9.0, "la": 22.0, "perturbation": 20.0}
# dram__bytes_read.sum + dram__bytes_write.sum of lav2_kernel, one `ncu --set full` capture (bytes per launch)
TRAFFIC = {"view14_hdr32_lav2": (7.67e6 + 3.07e6, "profiles/r2_lav2_view14_summary.md")}


def _clock_sampler(stop, samples, gpu_index):
    q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
    while not stop.is_set():
        try:
            out = subprocess.run(["nvidia-smi", f"--id={gpu_index}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                 capture_output=True, text=True, timeout=5).stdout.strip().splitlines()
            if out:
                samples.append([x.strip() for x in out[0].split(",")])
        except Exception:
            pass
        stop.wait(0.2)


def _clock_summary(samples):
    if not samples:
        return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
    sm = sorted(int(s[0]) for s in samples if s[0].isdigit())
    names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
    reasons = [n for i, n in enumerate(names) if any(len(s) > 2 + i and s[2 + i].lower().startswith("active") for s in samples)]
    return {"sm_mhz": sm[len(sm) // 2] if sm else None,
            "sm_max_mhz": int(samples[0][1]) if samples[0][1].isdigit() else None, "reasons": reasons,
            "samples": len(samples)}


class Workload:
    """Inputs of one named workload, produced by the in-tree generator (libfshost.so)."""

    def __init__(self, name):
        from fractalshark_b200 import RenderAlgorithm, traits
        from fractalshark_b200.host_inputs import BlaTable, LaTable, Orbit, View
        from fractalshark_b200.views import PRESETS
        spec = WORKLOADS[name]
        self.name, self.spec = name, spec
        self.alg = getattr(RenderAlgorithm, spec["alg"])
        self.traits = traits(self.alg)
        self.w, self.h = spec["w"], spec["h"]
        if "window" in spec:
            bounds, self.n_iter = spec["window"], spec["n_iter"]
            self.where = "window x[%s, %s] y[%s, %s]" % (bounds[0], bounds[2], bounds[1], bounds[3])
        else:
            p = PRESETS[spec["view"]]
            bounds, self.n_iter = (p.min_x, p.min_y, p.max_x, p.max_y), spec.get("n_iter") or p.num_iterations
            self.where = "view%d" % spec["view"]
        self.view = View(bounds[0], bounds[1], bounds[2], bounds[3], self.w, self.h)
        fam = self.traits.family
        self.coords = self.view.coords(self.traits.numeric, direct=(fam == "direct"))
        self.orbit = self.table = None
        self.gen_times = {"orbit_s": 0.0, "table_s": 0.0, "table_again_s": 0.0}
        if fam in ("lav2", "bla"):
            t0 = time.time()
            self.orbit = Orbit(self.view, self.traits.numeric, self.n_iter, True)
            t1 = time.time()
            self.table = LaTable(self.orbit, 4) if fam == "lav2" else BlaTable(self.orbit)
            t2 = time.time()
            # the first build of a process also starts the host thread pool; a view change in a running application does not
            again = []
            for _ in range(3):
                t3 = time.time()
                LaTable(self.orbit, 4) if fam == "lav2" else BlaTable(self.orbit)
                again.append(time.time() - t3)
            self.gen_times = {"orbit_s": t1 - t0, "table_s": t2 - t1, "table_again_s": min(again)}
        self.label = f"{self.where}_{spec['alg']}_{self.w}x{self.h}_aa1_u32_maxiter{self.n_iter}"

    def launch(self, r):
        fam = self.traits.family
        if fam == "lav2":
            return r.RenderPerturbLAv2(self.alg, self.coords, self.n_iter)
        if fam == "bla":
            return r.RenderPerturbBLA(self.alg, self.orbit, self.table, self.coords, self.n_iter)
        return r.Render(self.alg, self.coords, self.n_iter, 1)

    def prepare(self, r, generation=1):
        assert r.InitializeMemory(self.w, self.h, 1, iter_bytes=4) == 0
        if self.traits.family == "lav2":
            assert r.InitializePerturb(generation, self.orbit, 0, None, self.table) == 0


def roofline_of(wl, kinds, total_sum, ms, peaks, world=1):
    """FP-issue roofline of one workload from the executed-step counters of one launch."""
    from fractalshark_b200 import Numeric
    t = ms * 1e-3
    fam, num = wl.traits.family, wl.traits.numeric
    out = {"bound": "fp32_issue", "unit": "T FP32 instr/s", "peak": peaks["fp32"] * world / 1e12}
    if fam == "direct":
        # 6 FP instructions per iteration (FADD, 3 FFMA/DFMA, FMUL, FFMA of the bailout norm); every counted iteration is executed
        is64 = num == Numeric.F64
        peak = peaks["fp64"] if is64 else peaks["fp32"]
        ach = total_sum * 6.0 / t
        out.update({"bound": "fp64_issue" if is64 else "fp32_issue", "unit": "T FP64 instr/s" if is64 else "T FP32 instr/s",
                    "peak": peak * world / 1e12, "achieved": ach / 1e12, "frac": ach / (peak * world),
                    "instr_per_iteration": 6, "executed_steps_per_launch": float(total_sum)})
        return out
    steps = {k: int(kinds.get(k, 0)) for k in ("at", "la", "perturbation")}
    exec_steps = float(sum(steps.values()))
    out.update({"executed_steps_per_launch": exec_steps, "executed_steps_by_kind": steps,
                "skip_factor": total_sum / max(exec_steps, 1.0)})
    if fam == "lav2" and num == Numeric.HDR32:
        executed = sum(steps[k] * EXECUTED_FP32[k] for k in steps)
        credit = sum(steps[k] * REFERENCE_CREDIT[k] for k in steps)
        out.update({"achieved": executed / t / 1e12, "frac": executed / t / (peaks["fp32"] * world),
                    "executed_fp32_per_step": EXECUTED_FP32,
                    "reference_work_credit": {"per_step": REFERENCE_CREDIT, "achieved": credit / t / 1e12,
                                              "frac": credit / t / (peaks["fp32"] * world)}})
    else:
        # no per-instruction model of these kernels' steps: SURVEY.md 8(d) credits only (20 per HDRx32 perturbation /
        # BLA step, ~280 per 2x32 step), labelled as such
        per = 280.0 if num in (Numeric.X2_32, Numeric.HDR2X32) else 20.0
        credit = exec_steps * per
        out.update({"achieved": None, "frac": None,
                    "reference_work_credit": {"per_step": per, "achieved": credit / t / 1e12,
                                              "frac": credit / t / (peaks["fp32"] * world)}})
    return out


def measure_config(name, peaks, flush, steps=3):
    """One entry of the `configs` array: a BASELINE config measured on this GPU, device-timed, with the reference's own
    CUDA kernel (oracle/_ref, the checker) timed on the same inputs beside it."""
    import numpy as np
    import torch
    from fractalshark_b200.gpu_renderer import GPURenderer
    wl = Workload(name)
    r = GPURenderer(torch.cuda.current_device())
    wl.prepare(r)

    def one():
        flush.zero_()
        torch.cuda.synchronize()
        r.ClearMemory()
        rc = wl.launch(r)
        assert rc == 0, GPURenderer.ConvertErrorToString(rc)
        assert r.SyncComputeStream() == 0
        return r.LastRenderMs()

    one()
    ms = min(one() for _ in range(steps))
    r.EnableStepCounter(True)
    one()
    kinds = r.ReadStepCounters()
    r.EnableStepCounter(False)
    rc, iters, _, red = r.RenderCurrent(wl.n_iter)
    assert rc == 0
    entry = {"workload": wl.label, "baseline_config": wl.spec["config"], "ms": ms, "value": red["Sum"] / (ms * 1e-3),
             "unit": "pixel-iters/s", "sum_pixel_iters": red["Sum"],
             "inputs_untimed_s": wl.gen_times, "roofline": roofline_of(wl, kinds, red["Sum"], ms, peaks)}
    r.close()
    try:
        import ref_renderer
        if ref_renderer.available():
            rr = ref_renderer.RefGPURenderer()
            wl.prepare(rr)
            rms = []
            for _ in range(2):
                flush.zero_()
                torch.cuda.synchronize()
                rr.ClearMemory()
                assert wl.launch(rr) == 0
                assert rr.SyncComputeStream() == 0
                rms.append(rr.LastRenderMs())
            rc, ref_iters, _, ref_red = rr.RenderCurrent(wl.n_iter)
            a, b = iters[:wl.h, :wl.w].astype(np.int64), ref_iters[:wl.h, :wl.w].astype(np.int64)
            entry["reference_cuda_kernel"] = {"ms": min(rms), "speedup": min(rms) / ms, "pixels_exact_vs_ours": float((a == b).mean()),
                                              "max_abs_diff": int(np.abs(a - b).max())}
            rr.close()
    except Exception as e:  # the checker is optional here
        entry["reference_cuda_kernel"] = {"unavailable": repr(e)[:200]}
    return entry


def cpu_port_sample(wl, threads, stride):
    """Oracle CPU port of the GPU algorithm (the checker, timed as a baseline only) on a regular sub-grid."""
    import oracle_cpu
    t0 = time.time()
    iters, steps = oracle_cpu.render_lav2(wl.alg, wl.w, wl.h, wl.coords, wl.orbit, wl.table, wl.n_iter, rows=(0, wl.h),
                                          col_step=stride, row_step=stride, threads=threads)
    dt = time.time() - t0
    total = int(iters[0:wl.h:stride, 0:wl.w:stride].sum())
    return total / dt, dt, f"1 of every {stride} rows x 1 of every {stride} columns ({-(-wl.h // stride) * -(-wl.w // stride)} pixels, {dt:.1f} s)"


class ReferenceCpu:
    """The reference's own CPU renderer of the path (oracle/_ref/libref_host.so), or None when it is not built."""

    def __init__(self, wl):
        import ref_host
        self.ok = ref_host.available() and wl.traits.family == "lav2"
        if self.ok:
            self.wl = wl
            self.session = ref_host.RefLaTable(wl.orbit, 4, wl.n_iter, 0)

    def sample(self, stride, threads=0):
        wl = self.wl
        t0 = time.time()
        total, _ = self.session.cpu_lav2(wl.w, wl.h, wl.coords, wl.n_iter, row_step=stride, col_step=stride, threads=threads)
        dt = time.time() - t0
        return total / dt, dt, f"1 of every {stride} rows x 1 of every {stride} columns ({-(-wl.h // stride) * -(-wl.w // stride)} pixels, {dt:.1f} s)"

    def sized_stride(self, budget_s, probe_stride=240):
        """Sub-grid stride whose render takes about `budget_s` (cost is ~ proportional to the pixel count)."""
        _, probe_dt, _ = self.sample(probe_stride)
        want = probe_stride / max((budget_s / max(probe_dt, 1e-3)) ** 0.5, 1e-3)
        for k in (8, 10, 12, 16, 20, 24, 30, 40, 48, 60, 80, 120, 160, 240):
            if k >= want:
                return k
        return probe_stride


WHAT_THE_CPU_ARM_IS = ("Fractal::CalcCpuPerturbationFractalLAV2<u32, float, Disable> (Cpu32PerturbedBLAV2HDR, Fractal.cpp:2485-2691): "
                       "per-pixel loop restated on the reference's own types and compiled LAReference/ATInfo/HDRFloat code "
                       "(oracle/ref_host_harness.cpp), row claiming + std::thread x hardware_concurrency as in the reference. "
                       "Its counts differ from the Gpu* algorithms' by design (bailout 256; isLAStageInvalid has the opposite "
                       "sense, so it skips far less: SURVEY.md section 7)")


def run_reference_arm(args, rank):
    """Reference arm of this tier: the reference's CPU renderer of the path on the box's host cores (rank 0 only)."""
    if rank != 0:
        return
    import oracle_cpu
    wl = Workload(args.workload)
    threads = oracle_cpu.hardware_threads()
    ref = ReferenceCpu(wl) if wl.traits.family == "lav2" else None
    vals, times, sample = [], [], ""
    n_passes = max(args.warmup + args.steps, 1)
    if ref is not None and ref.ok:
        kind = "reference"
        stride = ref.sized_stride(180.0 / n_passes)
        fn = lambda: ref.sample(stride)
    else:
        kind = "port"
        _, probe_dt, _ = cpu_port_sample(wl, threads, 16)
        stride = next((k for k in (1, 2, 3, 4, 6, 8, 12) if probe_dt * 256.0 / (k * k) <= 180.0 / n_passes), 16)
        fn = lambda: cpu_port_sample(wl, threads, stride)
    for i in range(args.warmup + args.steps):
        v, dt, sample = fn()
        if i >= args.warmup:
            vals.append(v)
            times.append(dt)
    value = sum(vals) / len(vals)
    line = {"impl": "reference", "metric": metric_name(wl), "value": value, "unit": "pixel-iters/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * sum(times) / len(times),
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32+i32 (HDRx32)",
            "data": "synthetic (preset coordinates, orbit + LA table generated in-process)",
            "config": {"workload": wl.label, "l2": "n/a (CPU)"},
            "cpu_baseline": {"value": value, "unit": "pixel-iters/s", "cores": threads, "kind": kind, "sample": sample,
                             "what": WHAT_THE_CPU_ARM_IS if kind == "reference" else "oracle/oracle_cpu.cpp: CPU port of the GPU algorithm"},
            "e2e": {"value": value, "unit": "pixel-iters/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


DUMP_SEED = 20240607
DUMP_SAMPLE_BYTES = 32 << 20


def dump_outputs(out_dir, iters, red, width, height):
    """What the timed render hands its caller, as float64 .npy files: the reduction [Min, Max, Sum // 2^32, Sum % 2^32],
    every row's and column's sum of the iteration buffer, and the whole rows of a fixed, seeded sample of the frame (about
    32 MB) with their row numbers.  All exact: counts are below 2^32 and a row or column has fewer than 2^21 of them."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    frame = iters[:height, :width].astype(np.float64)
    n_rows = min(height, max(1, DUMP_SAMPLE_BYTES // (8 * width)))
    rows = np.sort(np.random.default_rng(DUMP_SEED).choice(height, size=n_rows, replace=False))
    arrays = {"reduction": np.array([red["Min"], red["Max"], red["Sum"] >> 32, red["Sum"] & 0xFFFFFFFF], dtype=np.float64),
              "row_sums": frame.sum(axis=1), "column_sums": frame.sum(axis=0),
              "sample_rows": rows.astype(np.float64), "iterations_sample_rows": frame[rows]}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def metric_name(wl):
    return f"pixel-iters/sec (device-timed) for {wl.where.replace('view', 'View ')} perturb+LA" if wl.traits.family != "direct" \
        else f"pixel-iters/sec (device-timed) for {wl.where} direct escape time"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the `configs` array (the other BASELINE configs)")
    ap.add_argument("--configs", default=None, help="comma-separated workload names for the `configs` array")
    ap.add_argument("--workload", default=None, choices=sorted(WORKLOADS), help="headline workload (default: View 14 HDRx32 LAv2)")
    ap.add_argument("--view", type=int, default=None, choices=[5, 14], help="shorthand: --view 5 = --workload view5_hdr32_lav2")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write the frame the last timed step rendered to DIR/<name>.npy (float64; see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.workload is None:
        args.workload = "view5_hdr32_lav2" if args.view == 5 else HEADLINE
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference_arm(args, rank)
        return

    import numpy as np
    import torch
    import torch.distributed as dist
    from fractalshark_b200.gpu_renderer import GPURenderer

    if not torch.cuda.is_available() or not GPURenderer.TestCudaIsWorking():
        raise SystemExit("bench.py: no CUDA device -- the render path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    from fractalshark_b200.host_inputs import ReplicatedInputs
    spec = WORKLOADS[args.workload]
    lav2 = spec["alg"].endswith("LAv2") or "LAv2" in spec["alg"]
    if world > 1 and not lav2:
        raise SystemExit("bench.py: N > 1 runs the LAv2 workloads (inputs replicated by broadcast); use --gpus 1 for the others")

    # ---- inputs: produced once on rank 0 (GMP orbit, LA table), replicated to the other ranks with NCCL broadcasts
    # of the packed blobs (north_star); receivers upload straight from the received host buffers -------------------
    bcast_ms = None
    wl = Workload(args.workload) if rank == 0 else None
    if lav2:
        if rank == 0:
            coords, orbit, la, n_iter, gen_times = wl.coords, wl.orbit, wl.table, wl.n_iter, wl.gen_times
        if world > 1:
            meta_box = [None]
            if rank == 0:
                meta, blobs = ReplicatedInputs.pack(coords, orbit, la, n_iter)
                meta["gen_times"] = gen_times
                meta["label"] = wl.label
                meta_box = [meta]
            dist.broadcast_object_list(meta_box, src=0)
            meta = meta_box[0]
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            dev = []
            for i, size in enumerate(meta["sizes"]):
                t = torch.from_numpy(blobs[i]).cuda() if rank == 0 else torch.empty(size, dtype=torch.uint8, device="cuda")
                dev.append(t)
            torch.cuda.synchronize()
            e0.record()
            for t in dev:
                if t.numel():
                    dist.broadcast(t, src=0)
            e1.record()
            torch.cuda.synchronize()
            bcast_ms = e0.elapsed_time(e1)
            if rank != 0:
                blobs = [t.cpu().numpy() for t in dev]
                coords, orbit, la, n_iter = ReplicatedInputs.unpack(meta, blobs)
                gen_times = meta["gen_times"]
            del dev
        else:
            meta, blobs = ReplicatedInputs.pack(coords, orbit, la, n_iter)
        # the e2e arm uploads from page-locked host memory: the same tables, copied once into pinned buffers
        pinned_blobs = []
        for b in blobs:
            t = torch.empty(max(int(b.size), 1), dtype=torch.uint8, pin_memory=True)
            t[:b.size] = torch.from_numpy(b)
            pinned_blobs.append(t.numpy()[:b.size])
        _, orbit_pinned, la_pinned, _ = ReplicatedInputs.unpack(meta, pinned_blobs)
    else:
        coords, orbit, la, n_iter, gen_times = wl.coords, wl.orbit, wl.table, wl.n_iter, wl.gen_times
    from fractalshark_b200 import RenderAlgorithm
    alg = getattr(RenderAlgorithm, spec["alg"])
    width, height = spec["w"], spec["h"]

    r = GPURenderer(local_rank)
    assert r.InitializeMemory(width, height, 1, iter_bytes=4) == 0
    assert r.SetShard(world, rank) == 0
    gen = 1
    if lav2:
        assert r.InitializePerturb(gen, orbit, 0, None, la) == 0
    assert r.SyncComputeStream() == 0
    launches0 = r.KernelLaunchCount()

    hp, wp = r.buffer_shape()
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")  # > 126 MB L2

    def launch():
        if lav2:
            return r.RenderPerturbLAv2(alg, coords, n_iter)
        return wl.launch(r)

    def step_resident():
        flush.zero_()
        torch.cuda.synchronize()
        r.ClearMemory()
        rc = launch()
        assert rc == 0, GPURenderer.ConvertErrorToString(rc)
        assert r.SyncComputeStream() == 0
        return r.LastRenderMs()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step_resident()

    # ---- timed region: K steps, device-timed ---------------------------------------------------------------
    stop, samples = threading.Event(), []
    sampler = threading.Thread(target=_clock_sampler, args=(stop, samples, local_rank), daemon=True)
    sampler.start()
    barrier()
    t_wall0 = time.time()
    kernel_ms = [step_resident() for _ in range(args.steps)]
    barrier()
    wall_s = time.time() - t_wall0
    launches_timed = r.KernelLaunchCount() - launches0 - args.warmup
    if args.dump_outputs:
        # untimed: the frame of the last timed step, assembled on rank 0 (disjoint rows, so SUM == gather)
        rc, last_iters, _, last_red = r.RenderCurrent(n_iter)
        assert rc == 0
        if world > 1:
            dev = torch.from_numpy(last_iters.view(np.int32)).cuda()
            dist.reduce(dev, dst=0, op=dist.ReduceOp.SUM)
            last_iters = dev.cpu().numpy().view(np.uint32)
            frame = last_iters[:height, :width]
            last_red = {"Min": int(frame.min()), "Max": int(frame.max()), "Sum": int(frame.astype(np.int64).sum())}
        if rank == 0:
            dump_outputs(args.dump_outputs, last_iters, last_red, width, height)
    # executed-step count for the roofline: one extra, untimed launch of the counting variant of the kernel
    r.EnableStepCounter(True)
    step_resident()
    kinds = r.ReadStepCounters()
    r.EnableStepCounter(False)
    stop.set()
    sampler.join()
    # the same frame with the AT cycle watch off (every pass of ATInfo::PerformAT executed, as the reference does and as
    # round 1 of this library did): untimed for `value`, reported inside `roofline` -- it is the configuration the
    # ">= 50 % of the FP32 issue peak" target of BASELINE.json was written against
    all_passes = None
    if lav2 and world == 1:
        assert r.SetAtCycleDetection(False) == 0
        step_resident()
        ms_all = min(step_resident() for _ in range(3))
        r.EnableStepCounter(True)
        step_resident()
        kinds_all = r.ReadStepCounters()
        r.EnableStepCounter(False)
        assert r.SetAtCycleDetection(True) == 0
        all_passes = (ms_all, kinds_all)

    rc, iters, _, red = r.RenderCurrent(n_iter)
    assert rc == 0
    local_sum = int(iters[:height, :width].sum())  # this rank's rows (others are zero)

    # ---- merge the iteration buffer on rank 0 (NCCL reduce of disjoint rows == gather) ----------------------
    total_sum, max_ms = local_sum, sum(kernel_ms)
    gather_ms = None
    if world > 1:
        dev_iters = torch.from_numpy(iters.view(np.int32)).cuda()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        dist.reduce(dev_iters, dst=0, op=dist.ReduceOp.SUM)
        e1.record()
        torch.cuda.synchronize()
        gather_ms = e0.elapsed_time(e1)
        t = torch.tensor([float(max_ms)], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        max_ms = float(t.item())
        s = torch.tensor([local_sum], device="cuda", dtype=torch.int64)
        dist.all_reduce(s, op=dist.ReduceOp.SUM)
        total_sum = int(s.item())
        es = torch.tensor([kinds["at"], kinds["la"], kinds["perturbation"]], device="cuda", dtype=torch.float64)
        dist.all_reduce(es, op=dist.ReduceOp.SUM)
        kinds = {"at": int(es[0].item()), "la": int(es[1].item()), "perturbation": int(es[2].item())}
        if rank == 0:
            merged = dev_iters.cpu().numpy().view(np.uint32)
            assert int(merged[:height, :width].astype(np.int64).sum()) == total_sum

    ms_per_step = max_ms / args.steps
    value = total_sum / (ms_per_step * 1e-3)

    # ---- e2e: public call sequence with host buffers (every step re-uploads orbit + LA, reads results) ------
    e2e = e2e_as_is = None
    if lav2:
        h2d = orbit.count * orbit.elem_bytes + la.num_las * la.las_elem_bytes + la.num_stages * 8 + la.at_bytes
        # N=1: the frame lands in a pinned buffer.  N>1: ONE host frame in POSIX shared memory, page-locked in every
        # rank; each rank copies just the 4-row bands it rendered into their place (fs_render_current_shard), so the
        # frame is assembled on the host with no collective and 1/N of the frame crosses each GPU's PCIe link.
        shm, frame_kind = None, "pinned"
        if world == 1:
            frame = torch.empty((hp, wp), dtype=torch.int32, pin_memory=True).numpy().view(np.uint32)
        else:
            from fractalshark_b200.sharding import SharedFrame
            name = "fsb200_frame_%s" % os.environ.get("MASTER_PORT", "0")
            shared_ok = [True]
            if rank == 0:
                try:
                    shm = SharedFrame(name, (hp, wp), np.uint32, create=True)
                except OSError:
                    shared_ok = [False]
            dist.broadcast_object_list(shared_ok, src=0)
            if shared_ok[0]:
                if rank != 0:
                    shm = SharedFrame(name, (hp, wp), np.uint32)
                frame = shm.array
                frame_kind = "shared memory frame every rank writes its bands into"
            else:  # no POSIX shared memory on this host: every rank keeps its bands in a pinned frame of its own
                frame = torch.zeros((hp, wp), dtype=torch.int32, pin_memory=True).numpy().view(np.uint32)
                frame_kind = "per-rank pinned frames (no shared memory on this host)"
            dist.barrier()
        # result sink: the kernel stores finished pixels into the host frame while it runs (fs_set_result_sink page-locks
        # and maps the frame if it is not yet), RenderCurrent then only fetches the 24-byte reduction.
        rc = r.SetResultSink(frame)
        assert rc == 0, GPURenderer.ConvertErrorToString(rc)
        frame_kind += "; streamed by the render kernel (result sink)"

        def step_e2e(g):
            rc = r.InitializePerturb(g, orbit_pinned, 0, None, la_pinned)
            assert rc == 0
            r.ClearMemory()
            assert r.RenderPerturbLAv2(alg, coords, n_iter) == 0
            if world == 1:
                rc, it, _, rd = r.RenderCurrent(n_iter, iters_out=frame)
            else:
                rc, rd = r.RenderCurrentShard(n_iter, frame)
            assert rc == 0
            return rd["Sum"]

        for _ in range(2):
            gen += 1
            step_e2e(gen)
        barrier()
        t0 = time.time()
        e2e_sum = 0
        for _ in range(args.steps):
            gen += 1
            e2e_sum = step_e2e(gen)
        barrier()
        e2e_s = (time.time() - t0) / args.steps
        assert e2e_sum == local_sum
        # untimed: one more step into a zeroed host frame -- what arrives there is the whole picture of THIS step
        if rank == 0 or shm is None:
            frame[:] = 0
        barrier()
        gen += 1
        step_e2e(gen)
        barrier()
        if shm is None and world > 1:
            assert int(frame[:height, :width].astype(np.int64).sum()) == local_sum
        elif rank == 0:
            assert int(frame[:height, :width].astype(np.int64).sum()) == total_sum
        if world > 1:
            t = torch.tensor([e2e_s], device="cuda", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            e2e_s = float(t.item())
            dist.barrier()
        assert r.SetResultSink(None) == 0
        if world > 1:
            del frame
            dist.barrier()
            if shm is not None:
                shm.close()
        # whole-job host<->device bytes per step: every rank uploads its own copy of the tables, the frame leaves once
        e2e = {"value": total_sum / e2e_s, "unit": "pixel-iters/s", "h2d_bytes_per_step": h2d * world,
               "d2h_bytes_per_step": hp * wp * 4 + 24 * world, "ms_per_step": e2e_s * 1e3, "host_frame": frame_kind,
               "inputs": "page-locked"}
        # the drop-in-as-is variant: pageable tables (what LAReference / PerturbationResults hand over today) and a
        # pageable frame copied after the render, as an unmodified caller would run it (N = 1)
        if world == 1:
            plain = np.empty((hp, wp), np.uint32)

            def step_as_is(g):
                assert r.InitializePerturb(g, orbit, 0, None, la) == 0
                r.ClearMemory()
                assert r.RenderPerturbLAv2(alg, coords, n_iter) == 0
                rc, it, _, rd = r.RenderCurrent(n_iter, iters_out=plain)
                assert rc == 0
                return rd["Sum"]

            for _ in range(2):
                gen += 1
                step_as_is(gen)
            torch.cuda.synchronize()
            t0 = time.time()
            for _ in range(args.steps):
                gen += 1
                s_as_is = step_as_is(gen)
            as_is_s = (time.time() - t0) / args.steps
            assert s_as_is == local_sum and int(plain[:height, :width].astype(np.int64).sum()) == total_sum
            e2e_as_is = {"value": total_sum / as_is_s, "unit": "pixel-iters/s", "ms_per_step": as_is_s * 1e3,
                         "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": hp * wp * 4 + 24,
                         "inputs": "pageable", "host_frame": "pageable; copied after the render"}
    else:
        # direct kernels have no table upload: e2e = coordinates in, frame out
        plain = torch.empty((hp, wp), dtype=torch.int32, pin_memory=True).numpy().view(np.uint32)
        for _ in range(2):
            r.ClearMemory(); launch(); r.RenderCurrent(n_iter, iters_out=plain)
        torch.cuda.synchronize()
        t0 = time.time()
        for _ in range(args.steps):
            r.ClearMemory()
            assert launch() == 0
            rc, it, _, rd = r.RenderCurrent(n_iter, iters_out=plain)
        e2e_s = (time.time() - t0) / args.steps
        e2e = {"value": total_sum / e2e_s, "unit": "pixel-iters/s", "h2d_bytes_per_step": 64, "d2h_bytes_per_step": hp * wp * 4 + 24,
               "ms_per_step": e2e_s * 1e3, "host_frame": "pinned; copied after the render"}

    # ---- time to the first frame of a new reference orbit: orbit + table (host, untimed above), upload, frame --------------
    first_frame = None
    if lav2:
        ups = []
        for _ in range(5):
            gen += 1
            torch.cuda.synchronize()
            t0 = time.time()
            assert r.InitializePerturb(gen, orbit_pinned, 0, None, la_pinned) == 0
            assert r.SyncComputeStream() == 0
            ups.append((time.time() - t0) * 1e3)
        first_frame = {"orbit_s": gen_times["orbit_s"], "table_s": gen_times["table_s"],
                       "table_again_s": gen_times.get("table_again_s"), "upload_ms": min(ups),
                       "frame_ms": ms_per_step,
                       "what": "reference orbit (in-tree GMP loop, three threads from 4,096 bits of precision) and LA table (in-tree builder, byte-identical to "
                               "the reference's) on the host, InitializePerturb from page-locked memory incl. the device-side "
                               "repacks, one frame"}

    # ---- roofline -----------------------------------------------------------------------------------------------
    peaks = {"fp32": GPURenderer.MeasureFp32IssuePeak(local_rank), "fp64": GPURenderer.MeasureFp64IssuePeak(local_rank)}
    if rank == 0:
        roofline = roofline_of(wl, kinds, total_sum, ms_per_step, peaks, world)
        if all_passes is not None:
            ra = roofline_of(wl, all_passes[1], total_sum, all_passes[0], peaks, world)
            roofline["every_at_pass_executed"] = {
                "ms_per_step": all_passes[0], "value": total_sum / (all_passes[0] * 1e-3),
                "executed_steps_by_kind": ra.get("executed_steps_by_kind"), "achieved": ra.get("achieved"), "frac": ra.get("frac"),
                "reference_work_credit_frac": (ra.get("reference_work_credit") or {}).get("frac"),
                "what": "same frame, same results, AT cycle watch off (fs_set_at_cycle_detection(0)): the kernel executes "
                        "every AT pass the reference executes"}
        traffic = TRAFFIC.get(args.workload)
        roofline["traffic"] = traffic[0] if traffic else None
        roofline["traffic_source"] = traffic[1] if traffic else None
        roofline["note"] = ("compute-bound scalar path (SURVEY.md 8d): not HBM, not tensor. achieved/frac = EXECUTED FP32-pipe "
                            "thread-instructions (device step counters x the instructions this kernel issues per step) / kernel "
                            "time / FFMA issue rate measured live by fs_measure_fp32_issue_peak on this GPU (MEASURED_PEAKS.json "
                            "has only HBM/bf16 peaks); reference_work_credit = the same steps at the reference formulation's work "
                            "per step.  The default build skips the AT passes of pixels whose passes have entered an exact "
                            "cycle (interior pixels: 97 % of the AT passes of this frame), so `frac` is over far fewer executed "
                            "FP32 instructions than the reference formulation needs; `every_at_pass_executed` is the same "
                            "frame with that shortcut off.")

        line = {"metric": metric_name(wl), "value": value, "unit": "pixel-iters/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong",
                "vs_baseline": None, "dtype": "f32+i32 (HDRx32)" if "HDRx32" in spec["alg"] else spec["alg"],
                "data": f"synthetic ({wl.where} coordinates; orbit via GMP + table generated in-process, untimed: "
                        f"{gen_times['orbit_s']:.3f}s + {gen_times['table_s']:.3f}s)",
                "config": {"workload": wl.label, "l2": "flushed between timed iterations (256 MiB memset)",
                           "sharding": f"4-row tile bands round-robin over {world} rank(s)",
                           "orbit_entries": orbit.count if orbit is not None else 0,
                           "la_records": getattr(la, "num_las", 0), "la_stages": getattr(la, "stage_count", 0)},
                "clocks": _clock_summary(samples),
                "e2e": e2e,
                "gpu_launches": int(launches_timed),
                "roofline": roofline,
                "peaks_measured_live": {"fp32_instr_per_s": peaks["fp32"], "fp64_instr_per_s": peaks["fp64"]},
                "wall_ms_per_step_incl_flush": wall_s * 1e3 / args.steps,
                "sum_pixel_iters": total_sum}
        if e2e_as_is is not None:
            line["e2e_as_is"] = e2e_as_is
        if first_frame is not None:
            line["time_to_first_frame"] = first_frame
        if gather_ms is not None:
            line["gather_ms"] = gather_ms
            line["input_broadcast_ms"] = bcast_ms

        # reference CUDA kernel (oracle/_ref, the checker) timed on the same GPU and inputs, for context
        try:
            import ref_renderer
            if ref_renderer.available() and world == 1:
                rr = ref_renderer.RefGPURenderer()
                wl.prepare(rr)
                ms = []
                for i in range(3):
                    flush.zero_()
                    torch.cuda.synchronize()
                    rr.ClearMemory()
                    assert wl.launch(rr) == 0
                    assert rr.SyncComputeStream() == 0
                    ms.append(rr.LastRenderMs())
                rc, ref_iters, _, ref_red = rr.RenderCurrent(n_iter)
                exact = float((ref_iters[:height, :width] == iters[:height, :width]).mean())
                line["reference_cuda_kernel"] = {"ms_per_step": min(ms[1:]), "value": ref_red["Sum"] / (min(ms[1:]) * 1e-3),
                                                 "unit": "pixel-iters/s", "pixels_exact_vs_ours": exact,
                                                 "what": "the reference's own kernel for this RenderAlgorithm, built for sm_100a"}
                rr.close()
        except Exception as e:  # the checker is optional here
            line["reference_cuda_kernel"] = {"unavailable": repr(e)[:200]}
        r.close()
        r = None

        # ---- the other BASELINE configs --------------------------------------------------------------------------
        if world == 1 and not args.no_configs:
            names = args.configs.split(",") if args.configs else [n for n in DEFAULT_CONFIGS if n != args.workload]
            line["configs"] = []
            for name in names:
                try:
                    line["configs"].append(measure_config(name, peaks, flush))
                except Exception as e:
                    line["configs"].append({"workload": name, "error": repr(e)[:300]})

        if not args.no_cpu_baseline and lav2:
            import oracle_cpu
            threads = oracle_cpu.hardware_threads()
            try:
                port_v, port_dt, port_sample = cpu_port_sample(wl, threads, 6 if spec.get("view") == 5 else 2)
                cb = {"value": port_v, "unit": "pixel-iters/s", "cores": threads, "kind": "port", "sample": port_sample,
                      "what": "oracle/oracle_cpu.cpp: CPU port of the GPU algorithm"}
            except NotImplementedError as e:  # numeric types the CPU port does not restate (2x32, HDRx64 ...)
                port_v, port_sample = None, None
                cb = {"value": None, "unit": "pixel-iters/s", "cores": threads, "kind": "port", "unavailable": str(e)[:200]}
            try:
                ref = ReferenceCpu(wl) if spec["alg"].startswith("GpuHDRx32") else None
                if ref is None:
                    raise RuntimeError("the reference CPU arm built here is the HDRFloat<float> LAv2 loop")
                if ref.ok:
                    stride = ref.sized_stride(15.0)
                    v, dt, sample = ref.sample(stride)
                    cb = {"value": v, "unit": "pixel-iters/s", "cores": threads, "kind": "reference", "sample": sample,
                          "what": WHAT_THE_CPU_ARM_IS,
                          "port": {"value": port_v, "sample": port_sample, "what": "oracle/oracle_cpu.cpp: CPU port of the GPU algorithm"}}
            except Exception as e:
                cb["reference_unavailable"] = repr(e)[:200]
            line["cpu_baseline"] = cb
        print(json.dumps(line), flush=True)
    if r is not None:
        r.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
