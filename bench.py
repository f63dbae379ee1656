#!/usr/bin/env python
"""bench.py — headline benchmark of the trace-and-shade hot path (BASELINE.json: Mrays/s and frames/s at 1920x1080).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--frames F] [--workload NAME] [--dump-outputs DIR]

One JSON line on stdout (rank 0).  A "step" is one pass of the hot path over one batch of F camera frames per GPU; every
timed loop (headline, e2e, copy-only ceiling and the `secondary` workloads) runs K steps.
Workload "config2" (default) is BASELINE.json configs[1]: the reference's default scene at 1920x1080, reflection depth
20 (Default::scrnshotRefections), 1 sample/pixel, default camera; the F frames of a step are successive frames of one
reference process (the randDir stream continues from frame to frame), so every frame is a full config-2 render.
With N > 1 the frames are sharded across ranks with no communication ("weak" scaling: F frames per GPU per step);
each rank first skips the random stream to its own frames exactly as the reference's stream would have advanced.

  value      whole-job Mrays/s with everything resident in HBM (device output buffer), CUDA-event timed, max over ranks
  e2e        the same metric through the C ABI with HOST buffers: scene + cameras re-uploaded and every frame's
             ARGB copied back to pinned host memory inside the timed region
  roofline   census flops of the frames (SURVEY §8d: 1301.7 flop/pixel) / K2 kernel time, against the FP32 peak
  cpu_baseline / --impl reference: the unmodified reference (oracle/_ref/ref_render_fast, the reference's own
             -Ofast flags) on this box's host cores, harness-parallel over rows because the reference has no threads
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
sys.dont_write_bytecode = True          # the tree may be read-only; the benchmark leaves nothing in it

W, H, DEPTH = 1920, 1080, 20
CENSUS_FLOP_PER_PIXEL = 1301.7          # SURVEY.md §8(d), config 2 (our own census build counts 1270.9, see DESIGN.md)
NCU_RAW_CSV = ("profiles/r2_final/prof_k_trace_small_raw.csv", "profiles/r1_final/prof_k_trace_small_raw.csv")   # ncu --set full, newest first
UNFUSED_SCALAR_CEILING_TFLOPS = 35.8    # measured: un-fused FMUL+FADD issue ceiling, scalar (35.8) or packed f32x2 on independent chains (36.6): profiles/microbench_r2.jsonl
RAYS_PER_FRAME_CANONICAL = 7493076      # oracle counters, config 2, seed 12345 (3.6136 rays/pixel); recomputed live when possible
METRIC = "Mrays/s at 1920x1080, default scene, reflection depth 20 (frames/s alongside)"
WORKLOAD = "config2: default scene 1920x1080, reflection depth 20, 1 sample/pixel, default camera; a step is frames_per_step successive frames (randDir stream continues)"
L2_NOTE = ("GPU arm: outputs larger than L2 (frames_per_step x 8.3 MB of ARGB written per step per GPU against the 126 MB L2), inputs are a <1 KB scene; "
           "CPU arm: not applicable")


def shared_config(frames):
    """the same `config` object in both arms' lines (the driver compares them)"""
    return {"workload": WORKLOAD, "width": W, "height": H, "depth": DEPTH, "frames_per_step": frames, "l2": L2_NOTE}


def ncu_dram_bytes_per_launch():
    """roofline.traffic: dram__bytes_read.sum + dram__bytes_write.sum of one k_trace_small launch, read from the committed
    `ncu --set full` raw page (profiles/), per launch; None when no capture is in the tree"""
    import csv
    for rel in NCU_RAW_CSV:
        path = os.path.join(ROOT, rel)
        if not os.path.exists(path):
            continue
        rows = list(csv.reader(open(path)))
        hdr, units = rows[0], rows[1]
        for vals in rows[2:]:
            kernel = vals[hdr.index("Kernel Name")]
            if "k_trace_small" not in kernel:
                continue
            total = 0.0
            for name in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                i = hdr.index(name)
                v = float(vals[i].replace(",", ""))
                scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}[units[i]]
                total += v * scale
            return int(total), rel
    return None, None


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--frames", type=int, default=32, help="frames per GPU per step")
    ap.add_argument("--workload", default="config2")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the configs 3 / 4 / 5 measurements of the `secondary` object")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the headline's last timed step rendered (rank 0's frames) to DIR/*.npy, see dump_outputs()")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and (a.impl != "ours" or a.workload != "config2"):
        ap.error("--dump-outputs applies to the headline workload (--impl ours --workload config2)")
    return a


DUMP_SAMPLE_PIXELS = 1 << 20


def dump_outputs(frames):
    """frames: the [F, H, W] ARGB (0x00RRGGBB) frames one step returns, as a device tensor.  The whole step is F x 24.9 MB as
    float32 channels, so what --dump-outputs stores is (<= 50 MB in all, float32, R, G, B in 0 ... 255):
      last_frame_rgb     [H, W, 3]  the step's last frame, whole
      step_sample_rgb    [N, 3]     pixels drawn from all F frames at a fixed seeded set of positions (N <= 2^20) ...
      step_sample_index  [N, 3]     ... and those positions: frame, row, column"""
    import numpy as np
    import torch

    def rgb(argb):
        return np.stack([(argb >> s) & 255 for s in (16, 8, 0)], axis=-1).astype(np.float32)

    F = frames.shape[0]
    pos = np.unique(np.random.default_rng(20261020).integers(0, F * H * W, DUMP_SAMPLE_PIXELS))
    flat = frames.reshape(-1)
    sample = flat[torch.from_numpy(pos).to(flat.device)].cpu().numpy()
    f, rest = np.divmod(pos, H * W)
    y, x = np.divmod(rest, W)
    return {"last_frame_rgb": rgb(frames[F - 1].cpu().numpy()), "step_sample_rgb": rgb(sample),
            "step_sample_index": np.stack([f, y, x], axis=-1).astype(np.float32)}


# ----------------------------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed regions (B200_PROFILING.md's clocks line).  The sampler
    starts before the warm-up (nvidia-smi needs ~0.2 s to produce its first line); only the lines whose timestamp falls
    inside a window opened by begin() and closed by end() are used."""
    Q = ("timestamp,index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.rows = []
        self.windows = []
        self.p = None
        self.idx = gpu_index

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "20"],
                                      stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.p = None

    def _read(self):
        for line in self.p.stdout:
            self.rows.append((time.time(), line.strip()))

    def begin(self):
        self.windows.append([time.time(), None])

    def end(self):
        self.windows[-1][1] = time.time()

    def stop(self):
        if not self.p:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.1)
        self.p.terminate()
        try:
            self.p.wait(timeout=2)
        except Exception:
            self.p.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        import datetime
        for t, r in self.rows:
            c = [x.strip() for x in r.split(",")]
            if len(c) < 10:
                continue
            try:   # nvidia-smi's own timestamp (local time); the pipe may deliver lines late
                t = datetime.datetime.strptime(c[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
            except ValueError:
                pass
            # a line describes the interval that ended when it was printed: accept it up to one period after a window closed
            if not any(w0 <= t <= (w1 if w1 is not None else t) + 0.03 for w0, w1 in self.windows):
                continue
            try:
                sm.append(float(c[2])); mx.append(float(c[3]))
            except ValueError:
                continue
            for n, v in zip(names, c[6:10]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "sampled": "nvidia-smi -lms 20, lines inside the two timed regions"}


def reference_cpu_run(binary, nproc, frames=1):
    """Harness-parallel run of the unmodified reference: nproc processes, interleaved rows, frames frames each.
    Returns wall seconds (max over processes of their own render time)."""
    from oracle import pyoracle as O
    exe = os.path.join(O.REF_DIR, binary)
    procs = []
    env = dict(os.environ, RFX_SEED="12345")
    t0 = time.perf_counter()
    for r in range(nproc):
        procs.append(subprocess.Popen([exe, "--size", str(W), str(H), "--refl", str(DEPTH), "--frames", str(frames),
                                       "--rows", str(nproc), str(r)], stdout=subprocess.PIPE, env=env, text=True))
    inner = []
    for p in procs:
        out = p.communicate()[0]
        inner.append(json.loads(out)["total_seconds"])
    wall = time.perf_counter() - t0
    return max(inner), wall


def canonical_rays_per_frame():
    """rays of one canonical config-2 frame (oracle counters) — deterministic for seed 12345"""
    try:
        from oracle import pyoracle as O
        from reflaxman_b200 import scenes as S
        r = O.OracleRender(S.default_scene(), W, H, seed=12345).render(S.default_camera(), DEPTH)
        return r.counters["rays"]
    except Exception:
        return RAYS_PER_FRAME_CANONICAL


# ----------------------------------------------------------------------------------------------------------------------
def run_reference(args):
    """--impl reference: the reference's own CPU implementation on the host cores; rank 0 only."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import pyoracle as O
    cores = os.cpu_count() or 1
    binary = "ref_render_fast"
    if not O.have_ref(binary):
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/%s was not built (needs the reference tree, RFX_REFERENCE_SRC, at build time)" % binary}))
        return
    rays = canonical_rays_per_frame()
    F = args.frames
    times = []
    for i in range(args.warmup + args.steps):
        t, _ = reference_cpu_run(binary, cores, frames=F)   # one step: the same F successive config-2 frames as the GPU arm's step
        if i >= args.warmup:
            times.append(t)
    total = sum(times)
    fps = len(times) * F / total
    val = fps * rays / 1e6
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": "Mrays/s", "frames_per_s": fps,
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": shared_config(F),
        "cpu_baseline": {"value": val, "unit": "Mrays/s", "cores": cores, "kind": "reference",
                         "sample": "%d frames per step; unmodified reference sources, reference flags -Ofast -fexpensive-optimizations (+NDEBUG), "
                                   "harness-parallel: %d processes x interleaved rows through Scene::trace (the reference itself is single-threaded); "
                                   "rays per frame = canonical config-2 count (%d)" % (F, cores, rays)},
        "e2e": {"value": val, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ----------------------------------------------------------------------------------------------------------------------
def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    from reflaxman_b200 import capi, scenes as S

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the hot path has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    F = args.frames
    K, Wm = args.steps, max(args.warmup, 3)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    t_create = time.perf_counter()
    ctx = capi.Context(local)                 # rfx_create: builds the 8.4 MB accept-count table of the LCG cycle (k_rng_table)
    ctx.synchronize()
    create_ms = 1e3 * (time.perf_counter() - t_create)
    if os.environ.get("RFX_COPY_STREAMS"):    # A/B knob of the e2e pipeline (tools/r2_session2.sh); default 1
        ctx.set_option("copy_streams", int(os.environ["RFX_COPY_STREAMS"]))
    scene = S.default_scene()
    ctx.load_scene(scene)
    ctx.set_image_size(W, H)
    ctx.set_seeds(12345, 12345)
    cam = S.default_camera()
    cams = capi.pack_cameras([cam] * F)
    info = ctx.device_info()

    # frame sharding: rank r owns frames [r * per_rank, (r+1) * per_rank) of the global sequence; skip the randDir stream there
    steps_total = 2 * (Wm + K) + 3
    per_rank = steps_total * F
    if rank > 0:
        ctx.skip_samples(rank * per_rank * W * H)
    ctx.synchronize()

    out_dev = torch.empty((F, H, W), dtype=torch.int32, device="cuda")      # F * 8.3 MB: larger than the 126 MB L2 for F >= 16
    out_host = torch.empty((F, H, W), dtype=torch.int32).pin_memory()
    stream = torch.cuda.Stream()            # explicit stream: our kernels and the timing events share it
    torch.cuda.set_stream(stream)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def maxreduce(x):
        if world > 1:
            t = torch.tensor([x], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return x

    def sumreduce(x):
        if world > 1:
            t = torch.tensor([x], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
            return float(t.item())
        return x

    # ---------------- device-resident arm ("value")
    for _ in range(Wm):
        ctx.render_frames_device(cams, DEPTH, 1, out_dev.data_ptr(), stream.cuda_stream)
    barrier()
    ctx.stats_reset()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    sampler.begin()
    e0.record(stream)
    for _ in range(K):
        ctx.render_frames_device(cams, DEPTH, 1, out_dev.data_ptr(), stream.cuda_stream)
    e1.record(stream)
    barrier()
    sampler.end()
    dumped = dump_outputs(out_dev) if args.dump_outputs and rank == 0 else None    # before the next render overwrites out_dev
    ms = maxreduce(e0.elapsed_time(e1))
    st = ctx.stats()
    rays_total = sumreduce(float(st["rays"]))
    launches = st["kernel_launches"]
    frames_total = K * F * world
    value = rays_total / (ms * 1e-3) / 1e6
    fps = frames_total / (ms * 1e-3)

    # ---------------- K2 kernel duration, live: one more step with every K2 launch bracketed by CUDA events on its stream
    ctx.enable_profiling(True)
    ctx.stats_reset()
    ctx.render_frames_device(cams, DEPTH, 1, out_dev.data_ptr(), stream.cuda_stream)
    torch.cuda.synchronize()
    stp = ctx.stats()
    ctx.enable_profiling(False)
    k2_ms_per_frame = stp["trace_kernel_ms"] / max(stp["trace_kernels"], 1)
    k2_share = stp["trace_kernel_ms"] / (ms / K)
    # the same with the tile-order history dropped before every frame: what the FIRST frame over a grid costs (index order),
    # and what an interactive front end whose renderNext slices never repeat pays on every launch
    ctx.enable_profiling(True)
    ctx.stats_reset()
    for f in range(min(F, 8)):
        ctx.set_tile_ordering(True)           # resets the history
        ctx.render_frames_device(cams[f:f + 1], DEPTH, 1, out_dev.data_ptr(), stream.cuda_stream)
    torch.cuda.synchronize()
    stc = ctx.stats()
    ctx.enable_profiling(False)
    k2_cold_ms = stc["trace_kernel_ms"] / max(stc["trace_kernels"], 1)

    # ---------------- end-to-end arm through the C ABI with host buffers
    def e2e_step():
        ctx.load_scene(scene)                         # host -> device: scene blob (+ textures when present)
        ctx.render_frames(cams, DEPTH, 1, out=out_host.numpy())   # cameras in, F ARGB frames back to pinned host memory
    for _ in range(Wm):
        e2e_step()
    barrier()
    ctx.stats_reset()
    sampler.begin()
    t0 = time.perf_counter()
    for _ in range(K):
        e2e_step()
    torch.cuda.synchronize()
    e2e_s = maxreduce(time.perf_counter() - t0)
    sampler.end()
    clocks = sampler.stop() if rank == 0 else None
    # copy-only ceiling of the same box, same buffers: F frames of 8.3 MB device -> pinned host per step on every rank at once, no
    # rendering.  e2e cannot exceed it; at 4-8 GPUs it is what binds (the host side of the box absorbs ~95 GB/s in total).
    def copy_step():
        for f in range(F):
            out_host[f].copy_(out_dev[f], non_blocking=True)
    for _ in range(2):
        copy_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(K):
        copy_step()
    torch.cuda.synchronize()
    copy_s = maxreduce(time.perf_counter() - t0)
    d2h_ceiling_fps = K * F * world / copy_s
    if world > 1:
        dist.barrier()
    st2 = ctx.stats()
    e2e_rays = sumreduce(float(st2["rays"]))
    e2e_value = e2e_rays / e2e_s / 1e6
    h2d = st2["h2d_bytes"] / K + cams.nbytes
    d2h = st2["d2h_bytes"] / K

    info = ctx.device_info()
    ctx.close()
    del out_dev
    torch.cuda.set_stream(torch.cuda.default_stream())
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    sm_max = float(peaks.get("sm_max_mhz", 1965.0))
    fp32_peak = 2 * 128 * info["sm_count"] * sm_max * 1e6 / 1e12          # FFMA peak, TFLOP/s (MEASURED_PEAKS.json has no FP32 entry)

    # ---------------- BASELINE.json configs[2..4] (every rank takes part; device-timed, max over ranks)
    secondary = None
    if not args.no_secondary:
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        import bench_extra
        env = bench_extra.Env()
        secondary = {"config3_split_8k_frame": bench_extra.config3(env, steps=K, warmup=3),
                     "config5_orbit_240_frames": bench_extra.config5(env, steps=K, warmup=3)}
        if world == 1:
            secondary["config4_1024_spheres_depth_sweep"] = bench_extra.config4(env, steps=K, fp32_peak_tflops=fp32_peak)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---------------- roofline (FP32 CUDA cores; this path is neither HBM- nor tensor-bound, SURVEY §8d)
    flops_per_frame = CENSUS_FLOP_PER_PIXEL * W * H
    achieved = flops_per_frame / (k2_ms_per_frame * 1e-3) / 1e12
    traffic, traffic_src = ncu_dram_bytes_per_launch()
    roofline = {"bound": "fp32", "achieved": achieved, "peak": fp32_peak, "unit": "TFLOP/s", "frac": achieved / fp32_peak,
                "traffic": traffic, "traffic_source": traffic_src,
                "kernel": "k_trace_small<0,false>", "kernel_ms_per_launch": k2_ms_per_frame, "kernel_share_of_step": k2_share,
                "kernel_ms_per_launch_cold": k2_cold_ms,
                "note": "bound is FP32 CUDA-core issue (neither hbm nor tensor: >= 80 flop per mandatory byte); traffic = dram__bytes_read+write of one "
                        "launch, read from the committed ncu --set full raw page (the 8.3 MB ARGB frame stays in the 126 MB L2 until evicted); "
                        "achieved = SURVEY census 1301.7 flop/pixel x 1920x1080 per launch / mean k_trace_small duration (CUDA events on its stream, "
                        "warm = tiles started in the cost order the previous frame recorded; cold = first frame over a grid); "
                        "peak = 2*128*SMs*sm_max_mhz (FFMA; MEASURED_PEAKS.json has no FP32 entry; microbench measured 70.4). The arithmetic "
                        "must stay un-fused for parity: FMUL+FADD tops out at 35.8 TFLOP/s scalar and 36.6 packed (FMUL2/FADD2 on independent chains; "
                        "a dependent packed pair is contracted into FFMA2 by ptxas even under --fmad=false): profiles/microbench_r2.jsonl, "
                        "tools/ffma2_contraction_repro.cu; first frame over a grid = middle tile rows first (no recording to replay)",
                "unfused_scalar_ceiling_tflops": UNFUSED_SCALAR_CEILING_TFLOPS, "frac_of_unfused_scalar_ceiling": achieved / UNFUSED_SCALAR_CEILING_TFLOPS}

    cpu = None
    if not args.no_cpu_baseline:
        try:
            from oracle import pyoracle as O
            cores = os.cpu_count() or 1
            if O.have_ref("ref_render_fast"):
                rays1 = canonical_rays_per_frame()
                t, _ = reference_cpu_run("ref_render_fast", cores, frames=1)
                t1, _ = reference_cpu_run("ref_render_fast", 1, frames=1)
                cpu = {"value": rays1 / t / 1e6, "unit": "Mrays/s", "cores": cores, "kind": "reference",
                       "sample": "one config-2 frame (1920x1080, depth 20); unmodified reference, reference flags -Ofast; harness-parallel over "
                                 "%d processes (interleaved rows via Scene::trace)" % cores,
                       "single_thread_value": rays1 / t1 / 1e6, "frames_per_s": 1.0 / t, "single_thread_frames_per_s": 1.0 / t1}
        except Exception as ex:   # the baseline is a report, not the product
            cpu = {"value": None, "unit": "Mrays/s", "cores": 0, "kind": "reference", "sample": "failed: %r" % (ex,)}

    line = {
        "metric": METRIC, "value": value, "unit": "Mrays/s", "frames_per_s": fps,
        "n_gpus": world, "steps": K, "warmup": Wm, "ms_per_step": ms / K,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": shared_config(F),
        "frames_per_step_per_gpu": F, "rays_per_frame": rays_total / frames_total,
        "e2e": {"value": e2e_value, "unit": "Mrays/s", "frames_per_s": frames_total / e2e_s, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                "d2h_copy_only_frames_per_s": d2h_ceiling_fps, "d2h_copy_only_GBps": d2h_ceiling_fps * W * H * 4 / 1e9,
                "frac_of_d2h_ceiling": (frames_total / e2e_s) / d2h_ceiling_fps, "frac_of_device_resident": e2e_value / value,
                "binds": "device->host copies (box ceiling)" if (frames_total / e2e_s) / d2h_ceiling_fps > 0.85 else "rendering"},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "roofline": roofline,
        "cpu_baseline": cpu,
        "secondary": secondary,
        "context_create_ms": create_ms,
        "device": info["name"],
    }
    print(json.dumps(line))
    if dumped is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in dumped.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    elif a.workload in ("config3", "config4", "config5"):
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        import bench_extra
        bench_extra.main(a)
    else:
        run_ours(a)
