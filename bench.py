#!/usr/bin/env python
"""bench.py — Mray/s of the ToyPathTracer hot path (DrawTest -> Trace/HitWorld/Scatter) on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--mode fast|exact] [--dump-outputs DIR]

Workload (BASELINE.json configs[1]): the reference's 46-sphere scene, 1280x720, 4 spp per frame, flags = 0
(non-progressive: every frame is a fresh image, BASELINE "DO_PROGRESSIVE off"). One STEP = one frame = one DrawTest
call of the reference (UpdateTest + DrawTest): ~16.8 M rays (camera + bounce + shadow, Test.cpp:122,199).

  value   whole-job Mray/s with the image resident in HBM: rays of the K timed steps / device time of those steps
          (CUDA events on the launching stream, one pair per step, summed; L2 flushed between steps, flush not
          timed), max over ranks.
  e2e     the same metric through the drop-in C-ABI with HOST buffers: per step tpt_set_scene (scene H2D, what
          UpdateTest+GetSceneDesc+UpdateSubresource do in the reference's GPU shells, TestWin.cpp:258-283; the
          option "scene_upload_always" makes it a real copy every step although the bytes do not change) +
          tpt_draw (kernel, image and ray count into pinned host memory), wall clock around the synchronous call.
  N > 1   north_star's tiled image split, weak scaling: step s renders the N frames s*N .. s*N+N-1 of ONE 1280x720
          image (accumulated with kFlagProgressive); rank r traces rows r, r+N, ... of all N frames (rows are the
          independent RNG chains, Test.cpp:278-280) into its packed band, then ONE all_gather per step assembles the
          14.7 MB image on every rank — inside the timed region. One frame's worth of rays per GPU per step at every N.
          `strong` sub-record: BASELINE configs[3] (3840x2160, 64 spp, one image split over the N GPUs) with the 1-GPU
          time of the same image, assembled A) by NCCL all_gather, B) by the tile kernel's peer stores over NVLink.

--impl reference times the UNMODIFIED reference C++ path (oracle/_ref/libtoyref.so, enkiTS on all host threads)
on the same workload; rank 0 only.

--dump-outputs DIR writes the float32 RGBA image of the last timed step (1280x720x4; at N > 1 the assembled image)
to DIR/image.npy from rank 0. Which frames that step renders depends only on W (at least 3), K and N, so two builds
run with the same arguments can be compared image for image. At N = 1 it is frame W+K-1 alone, which --mode exact and
--impl reference render bit for bit like the reference; the fast mode adds its samples with float atomics, so two of
its runs agree to rounding, not bit for bit.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

W, H, SPP = 1280, 720, 4
WORKLOAD = "46-sphere reference scene, 1280x720, 4 spp/frame, flags=0 (BASELINE configs[1]); step = one frame (one DrawTest)"
SPHERES = 46
FP32_TESTS_PER_S_PEAK = 148 * 128 * 1.965e9 / 17.0   # SURVEY §8d: ~16 FP32 ops + compare per ray-sphere test, no FMA


def load_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum of the dominant kernel from the committed ncu --set full capture
    (per launch, same workload); None when no capture of this round's kernel is committed."""
    try:
        for rnd in ("r02", "r01"):
            path = os.path.join(ROOT, "profiles", rnd, "ncu_traffic.json")
            if os.path.exists(path):
                return json.load(open(path)).get("k_fast_queue_1280x720_4spp_dram_bytes")
    except Exception:
        pass
    return None


def load_peaks():
    try:
        p = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks/throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "50",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) >= 7:
                self.rows.append(parts)

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if r[1].replace(".", "").isdigit()]
        reasons = []
        for name, col in (("hw_slowdown", 3), ("hw_thermal_slowdown", 4), ("sw_thermal_slowdown", 5), ("sw_power_cap", 6)):
            if any(r[col].lower().startswith("active") for r in self.rows):
                reasons.append(name)
        busy = [s for s in sm if s > 300] or sm
        return {"sm_mhz": statistics.median(busy) if busy else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def dump_outputs(directory, **arrays):
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, f"{name}.npy"), np.ascontiguousarray(a, dtype=np.float32))


def run_reference(args, rank):
    """The reference's own CPU implementation on the host cores (its enkiTS scheduler uses every hardware thread,
    Cpp/Source/enkiTS/TaskScheduler.cpp:1301). One step = one 1280x720 4-spp frame, like ours."""
    if rank != 0:
        return
    from oracle import pyoracle
    if not pyoracle.have_ref():
        pyoracle.build()
    kind = "reference" if pyoracle.have_ref() else "port"
    cores, cpu_info = usable_cores()
    buf = np.zeros((H, W, 4), np.float32)
    if kind == "reference":
        render = lambda f0, n: pyoracle.ref_render(W, H, f0, n, flags=0, buf=buf, want_seconds=True)[1:]
    else:
        import toypathtracer_b200 as tpt
        sph, mats, cam, em = tpt.reference_scene(W, H)
        render = lambda f0, n: (lambda r: (r[1], r[3]))(pyoracle.orc_render(sph, mats, cam, W, H, f0, n, flags=0, buf=buf, want_seconds=True))
    render(0, max(2, args.warmup))            # first frames pay thread spin-up (SURVEY §6)
    rays, secs = render(args.warmup, args.steps)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, image=buf)
    total_s = sum(secs)
    value = sum(rays) / total_s / 1e6
    line = {"impl": "reference", "metric": "Mray/s on 46-sphere scene @1280x720", "value": value, "unit": "Mray/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total_s / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "mode": "reference C++ SIMD path (enkiTS, all hardware threads)", "parallelism": "host CPU",
                       "l2": None, "timing": "steady clock around UpdateTest+DrawTest per frame", "threads": os.cpu_count()},
            "cpu_baseline": {"value": value, "unit": "Mray/s", "cores": cores, "kind": kind, "host": cpu_info,
                             "sample": f"{args.steps} frames of 1280x720x4spp after {max(2, args.warmup)} warm-up frames, "
                                       "UpdateTest+DrawTest per frame, steady clock"},
            "e2e": {"value": value, "unit": "Mray/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def cpu_baseline_sample():
    """Bounded sample of the reference CPU path on this box's host cores (rank 0, N=1 only): ~10-20 s."""
    from oracle import pyoracle
    kind = "reference" if pyoracle.have_ref() else "port"
    cores, cpu_info = usable_cores()
    buf = np.zeros((H, W, 4), np.float32)
    if kind == "reference":
        run = lambda f0, n: pyoracle.ref_render(W, H, f0, n, flags=0, buf=buf, want_seconds=True)[1:]
    else:
        import toypathtracer_b200 as tpt
        sph, mats, cam, em = tpt.reference_scene(W, H)
        run = lambda f0, n: (lambda r: (r[1], r[3]))(pyoracle.orc_render(sph, mats, cam, W, H, f0, n, flags=0, buf=buf, want_seconds=True))
    run(0, 3)
    t0 = time.time()
    rays, secs, frames = [], [], 0
    while time.time() - t0 < 12.0 and frames < 240:
        r, s = run(3 + frames, 8)
        rays += r; secs += s; frames += 8
    # median frame (BASELINE.md §3: discard warm-up, median of >= 30 frames)
    per_frame = sorted(r / s / 1e6 for r, s in zip(rays, secs))
    return {"value": per_frame[len(per_frame) // 2], "unit": "Mray/s", "cores": cores, "kind": kind, "host": cpu_info,
            "threads_spawned": os.cpu_count(),
            "sample": f"median of {frames} frames of 1280x720x4spp (UpdateTest+DrawTest each) after 3 warm-up frames; "
                      f"mean {sum(rays) / sum(secs) / 1e6:.1f} Mray/s"}


def host_cpu_info():
    """What the CPU arm can really use on this box: os.cpu_count() reports the machine, not the lease."""
    info = {"os_cpu_count": os.cpu_count()}
    try:
        info["sched_affinity"] = len(os.sched_getaffinity(0))
    except Exception:
        info["sched_affinity"] = None
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            info["cgroup_cpu_max"] = open(path).read().strip()
            break
        except Exception:
            info["cgroup_cpu_max"] = None
    try:
        info["loadavg"] = os.getloadavg()[0]
    except Exception:
        pass
    return info


def usable_cores():
    info = host_cpu_info()
    n = info.get("sched_affinity") or info["os_cpu_count"] or 1
    q = info.get("cgroup_cpu_max")
    if q:
        parts = q.split()
        try:
            if len(parts) == 2 and parts[0] != "max":
                n = min(n, max(1, int(float(parts[0]) / float(parts[1]) + 0.5)))
            elif len(parts) == 1 and int(parts[0]) > 0:
                n = min(n, max(1, int(int(parts[0]) / 100000 + 0.5)))
        except Exception:
            pass
    return n, info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=500)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--mode", default="fast", choices=["fast", "exact"])
    ap.add_argument("--variant", type=int, default=-1, help="fast kernel variant (default: library default)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-strong", action="store_true", help="skip the 3840x2160x64spp strong-scaling sub-record (N > 1)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's image as DIR/image.npy (float32)")
    args = ap.parse_args()
    if args.warmup < 3:
        args.warmup = 3

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank)
        return

    import torch
    import torch.distributed as dist
    import toypathtracer_b200 as tpt
    from toypathtracer_b200 import multigpu as mg

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    ctx = tpt.Context(local_rank)
    sph, mats, cam, em = tpt.reference_scene(W, H)
    ctx.set_scene(sph, mats, cam, em)
    if args.variant >= 0:
        ctx.set_option("fast_variant", args.variant)
    mode = tpt.MODE_FAST if args.mode == "fast" else tpt.MODE_EXACT
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)      # > 126 MB L2
    stream = torch.cuda.Stream(dev)          # a real (non-NULL) stream: the library treats NULL as "my own stream"
    torch.cuda.set_stream(stream)
    sh = stream.cuda_stream

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # N = 1: one frame per step, flags = 0 (the reference step). N > 1: north_star's tiled image split — step s renders
    # the N frames s*N .. s*N+N-1 of ONE 1280x720 image (accumulated with kFlagProgressive, every sample contributes),
    # rank r traces rows r, r+N, ... of all N frames into its packed band, and ONE all_gather per step assembles the
    # 14.7 MB image on every rank inside the timed region. Per-GPU work per step is one frame's worth at every N.
    row0, nrows, rstep = mg.rows_of_rank(H, rank, world)
    if world == 1:
        image = torch.zeros((H, W, 4), dtype=torch.float32, device=dev)
    else:
        band = torch.zeros((nrows, W, 4), dtype=torch.float32, device=dev)
    assembled = [None]

    def step(s, evs=None):
        flush.fill_(s & 0xFF)                                             # L2 flush, outside the timed events
        if evs is not None:
            evs[0].record(stream)
        if world == 1:
            ctx.draw(s, 1, W, H, image, flags=0, mode=mode, stream=sh, want_rays=False)
            if evs is not None:
                evs[1].record(stream)
        else:
            ctx.draw(s * world, world, W, H, band, flags=tpt.kFlagProgressive, mode=mode, rows=(row0, nrows, rstep, 1),
                     stream=sh, want_rays=False)
            if evs is not None:
                evs[1].record(stream)
            assembled[0] = mg.gather_rows(band, H, rank, world)           # the exchange step, every step
        if evs is not None:
            evs[2].record(stream)

    for s in range(args.warmup):
        step(s)
    ctx.read_ray_count(sh)                                                # reset the accumulated counter
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()                                                   # BEFORE the barrier: no rank enters the timed region late
        time.sleep(0.2)
    barrier()
    evs = [tuple(torch.cuda.Event(enable_timing=True) for _ in range(3)) for _ in range(args.steps)]
    wall0 = time.perf_counter()
    for s in range(args.steps):
        step(args.warmup + s, evs[s])
    barrier()
    wall = time.perf_counter() - wall0
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, image=(image if world == 1 else assembled[0]).cpu().numpy())
    step_ms = [a.elapsed_time(c) for a, b, c in evs]
    kernel_step_ms = [a.elapsed_time(b) for a, b, c in evs]
    exchange_ms = [b.elapsed_time(c) for a, b, c in evs]
    my_ms = sum(step_ms)
    dev_ms = my_ms
    rays = ctx.read_ray_count(sh)
    launches = ctx.last_launch_count() * args.steps
    per_rank_ms = [my_ms]

    if world > 1:
        t = torch.tensor([my_ms], dtype=torch.float64, device=dev)
        allt = torch.zeros(world, dtype=torch.float64, device=dev)
        dist.all_gather_into_tensor(allt, t)
        per_rank_ms = [float(x) for x in allt.cpu()]
        dev_ms = max(per_rank_ms)
        rays = mg.sum_ray_counts(rays, dev)
        lt = torch.tensor([launches], dtype=torch.int64, device=dev); dist.all_reduce(lt); launches = int(lt.item())

    # ---- end to end through the C-ABI (every rank; the slowest rank's wall time counts)
    e2e_steps = min(args.steps, 50)
    scene_bytes = 46 * 20 + 46 * 36 + 88 + 2 * 4
    if world == 1:
        # host backbuffer in, host backbuffer out: what a reference shell does per frame
        host = torch.zeros((H, W, 4), dtype=torch.float32).pin_memory().numpy()
        # every step carries its host -> device copy: by default tpt_set_scene skips the upload when the bytes are the
        # resident scene's (a shell calls UpdateTest every frame), which would leave this loop without any H2D
        ctx.set_option("scene_upload_always", 1)
        for s in range(3):
            ctx.set_scene(sph, mats, cam, em)
            ctx.draw(s, 1, W, H, host, flags=0, mode=mode)
        t0 = time.perf_counter()
        e2e_rays = 0
        upload = 0
        for s in range(e2e_steps):
            ctx.set_scene(sph, mats, cam, em)                              # scene H2D (UpdateTest + upload of the packed blob)
            upload += ctx.last_scene_upload_bytes()
            e2e_rays += ctx.draw(args.warmup + s, 1, W, H, host, flags=0, mode=mode)  # kernel + image D2H + count D2H
        e2e_s = time.perf_counter() - t0
        ctx.set_option("scene_upload_always", 0)
        h2d = upload // e2e_steps + (W * H * 16 if mode == tpt.MODE_EXACT else 0)  # packed blob; exact mode also uploads prev (bit parity)
        d2h = W * H * 16 + 8
        e2e_api = "tpt_set_scene + tpt_draw(host backbuffer) per step, wall clock"
    else:
        # per step: scene H2D on every rank, tpt_draw of the rank's rows (band resident in HBM: it is the accumulation
        # state, not a per-step input), all_gather, and rank 0 reads the assembled image + every rank its ray count back
        host = torch.zeros((H, W, 4), dtype=torch.float32).pin_memory()
        band.zero_()
        ctx.set_option("scene_upload_always", 1)      # a real scene H2D on every rank, every step (see the 1-GPU leg)
        upload = [0]
        def e2e_step(s):
            ctx.set_scene(sph, mats, cam, em)
            upload[0] = ctx.last_scene_upload_bytes()
            r = ctx.draw(s * world, world, W, H, band, flags=tpt.kFlagProgressive, mode=mode, rows=(row0, nrows, rstep, 1), stream=sh)
            img = mg.gather_rows(band, H, rank, world)
            if rank == 0:
                host.copy_(img, non_blocking=True)
            stream.synchronize()
            return r
        for s in range(3):
            e2e_step(s)
        barrier()
        t0 = time.perf_counter()
        e2e_rays = 0
        for s in range(e2e_steps):
            e2e_rays += e2e_step(3 + s)
        barrier()
        e2e_s = time.perf_counter() - t0
        t = torch.tensor([e2e_s], dtype=torch.float64, device=dev); dist.all_reduce(t, op=dist.ReduceOp.MAX); e2e_s = float(t.item())
        e2e_rays = mg.sum_ray_counts(e2e_rays, dev)
        ctx.set_option("scene_upload_always", 0)
        h2d = upload[0] * world
        d2h = W * H * 16 + 8 * world
        e2e_api = ("per step and rank: tpt_set_scene + tpt_draw(rows rank::N of N frames, device band) + all_gather; "
                   "rank 0 copies the assembled image to pinned host memory; wall clock, max over ranks")

    strong = None
    if world > 1 and args.mode == "fast" and not args.no_strong:
        strong = strong_scaling_record(ctx, tpt, mg, torch, dist, dev, stream, rank, world)

    if rank == 0:
        hbm_peak, peak_src = load_peaks()
        value = rays / (dev_ms * 1e-3) / 1e6
        kms = statistics.mean(kernel_step_ms)
        alg_bytes = (W * H * 16 + (W * H * 4 if world == 1 else W * H * 16)) // world   # float4 written (+ alpha / prev read)
        achieved = alg_bytes / (kms * 1e-3) / 1e9
        tests_per_s = (rays / world / args.steps) * (SPHERES + 2) / (kms * 1e-3)   # 48 padded spheres swept per ray
        line = {
            "metric": "Mray/s on 46-sphere scene @1280x720", "value": value, "unit": "Mray/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dev_ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "mode": args.mode,
                       "parallelism": (f"image rows interleaved over {world} GPUs, {world} frames per step accumulated "
                                       f"(kFlagProgressive), all_gather of the 14.7 MB image every step") if world > 1 else "1 GPU",
                       "l2": "flushed between steps (256 MiB fill), not timed",
                       "timing": "CUDA events per step on the launching stream (draw + exchange), summed; max over ranks",
                       "threads": None},
            "clocks": clocks,
            "per_rank_ms": per_rank_ms,
            "exchange_ms_per_step": statistics.mean(exchange_ms) if world > 1 else 0.0,
            "kernel_ms_per_step": kms,
            "e2e": {"value": e2e_rays / e2e_s / 1e6, "unit": "Mray/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "steps": e2e_steps, "ms_per_step": 1e3 * e2e_s / e2e_steps, "api": e2e_api},
            "gpu_launches": launches,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak,
                         "traffic": load_traffic() if args.mode == "fast" else None, "peak_source": peak_src,
                         "kernel": "k_fast_queue" if args.mode == "fast" else "k_trace_exact",
                         "algorithmic_bytes_per_launch": alg_bytes,
                         "note": "the path is FP32-issue bound, not HBM bound (SURVEY §8d): 16 B/pixel written per launch; "
                                 "see fp32 for the binding roofline",
                         "fp32": {"sphere_tests_per_s": tests_per_s, "peak_tests_per_s": FP32_TESTS_PER_S_PEAK,
                                  "frac": tests_per_s / FP32_TESTS_PER_S_PEAK,
                                  "peak_def": "148 SM x 128 lanes x 1.965 GHz / 17 FP32 issue slots per test (no FMA)"}},
            "wall_s": wall,
        }
        if strong is not None:
            line["strong"] = strong
        if world == 1 and args.mode == "fast":
            # the bit-exact mode on the same step, for the record (same API, same buffers; latency-bound: one serial RNG
            # chain per image row, Test.cpp:280)
            ex_steps = 8
            for s_ in range(2):
                ctx.draw(s_, 1, W, H, image, flags=0, mode=tpt.MODE_EXACT, stream=sh, want_rays=False)
            ctx.read_ray_count(sh)
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record(stream)
            for s_ in range(ex_steps):
                ctx.draw(2 + s_, 1, W, H, image, flags=0, mode=tpt.MODE_EXACT, stream=sh, want_rays=False)
            ev1.record(stream)
            torch.cuda.synchronize(dev)
            ex_rays = ctx.read_ray_count(sh)
            ex_ms = ev0.elapsed_time(ev1)
            line["exact_mode"] = {"value": ex_rays / ex_ms / 1e3, "unit": "Mray/s", "ms_per_step": ex_ms / ex_steps, "steps": ex_steps,
                                  "note": "TPT_MODE_EXACT: pixels and ray counts bit-identical to the reference CPU path; one frame "
                                          "traced per call (720 serial RNG chains: latency-bound)"}
            # the same calls with frame lookahead: a cache miss traces 16 consecutive frames in one launch, the next 15
            # one-frame calls only blend their cached frame (same bits, same counts; amortised over 32 calls = 2 misses)
            ctx.set_option("exact_lookahead", 16)
            for s_ in range(16):
                ctx.draw(100 + s_, 1, W, H, image, flags=0, mode=tpt.MODE_EXACT, stream=sh, want_rays=False)
            ctx.read_ray_count(sh)
            ev0.record(stream)
            for s_ in range(32):
                ctx.draw(116 + s_, 1, W, H, image, flags=0, mode=tpt.MODE_EXACT, stream=sh, want_rays=False)
            ev1.record(stream)
            torch.cuda.synchronize(dev)
            la_rays = ctx.read_ray_count(sh)
            la_ms = ev0.elapsed_time(ev1)
            ctx.set_option("exact_lookahead", 0)
            line["exact_mode_lookahead16"] = {"value": la_rays / la_ms / 1e3, "unit": "Mray/s", "ms_per_step": la_ms / 32, "steps": 32,
                                              "note": "exact_lookahead = 16: amortised over 32 one-frame calls (2 trace launches of 16 "
                                                      "frames + 32 blends); first-call latency = 16 frames"}
            # the drop-in's default (exact_lookahead = -1, adaptive): a fresh sequence of 64 one-frame calls INCLUDING the
            # ramp-up (windows of 1, 2, 4, 8, 16, 16, 16 frames, then 1 frame of the next window of 16 -> 79 frames traced for
            # 64 served; ray counts are those of the 64 frames handed out)
            ctx.set_option("exact_lookahead", -1)
            ev0.record(stream)
            for s_ in range(64):
                ctx.draw(1000 + s_, 1, W, H, image, flags=0, mode=tpt.MODE_EXACT, stream=sh, want_rays=False)
            ev1.record(stream)
            torch.cuda.synchronize(dev)
            ad_rays = ctx.read_ray_count(sh)
            ad_ms = ev0.elapsed_time(ev1)
            ctx.set_option("exact_lookahead", 0)
            line["exact_mode_adaptive"] = {"value": ad_rays / ad_ms / 1e3, "unit": "Mray/s", "ms_per_step": ad_ms / 64, "steps": 64,
                                           "note": "exact_lookahead = -1 (what libtoytest_b200.so's DrawTest uses): 64 consecutive "
                                                   "one-frame calls from a cold start, window doubling 1..16; no first-call latency"}
        if world == 1 and args.mode == "fast":
            # the reference-GPU-compatible estimator (per-pixel seeds, ComputeShader.hlsl) on the same frame: like for like
            # with the numbers the reference publishes for its own GPU back-ends (readme.md:64-77, other hardware)
            rg = {}
            for name, m in (("strict", tpt.MODE_REFGPU), ("native", tpt.MODE_REFGPU_FAST)):
                for s_ in range(2):
                    ctx.draw(s_, 1, W, H, image, flags=0, mode=m, stream=sh, want_rays=False)
                ctx.read_ray_count(sh)
                ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                ev0.record(stream)
                for s_ in range(10):
                    ctx.draw(2 + s_, 1, W, H, image, flags=0, mode=m, stream=sh, want_rays=False)
                ev1.record(stream)
                torch.cuda.synchronize(dev)
                rg[name] = {"value": ctx.read_ray_count(sh) / ev0.elapsed_time(ev1) / 1e3, "unit": "Mray/s", "ms_per_step": ev0.elapsed_time(ev1) / 10}
            rg["note"] = ("TPT_MODE_REFGPU / _FAST: the estimator of Cpp/Windows/ComputeShader.hlsl; the reference's readme.md reports "
                          "3920 Mray/s (D3D11, GeForce RTX 3080 Ti) and 1680 Mray/s (Metal, M4 Max) for its own GPU paths on this workload")
            line["refgpu_mode"] = rg
        if world == 1 and not args.no_cpu_baseline:
            try:
                line["cpu_baseline"] = cpu_baseline_sample()
            except Exception as ex:  # the oracle is a checker; its absence must not hide the GPU number
                line["cpu_baseline"] = {"error": str(ex)}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def strong_scaling_record(ctx, tpt, mg, torch, dist, dev, stream, rank, world):
    """BASELINE configs[3]: ONE 3840x2160 image at 64 spp (frames 0..15), rows interleaved over the ranks.
      one_gpu_ms  rank 0 renders the whole image alone (the other ranks idle)
      A           every rank renders its packed band (k_fast_queue) + ONE NCCL all_gather assembles it on every rank
      B           every rank's tile kernel (k_fast_tileq) stores its finished tiles straight into rank 0's image over
                  NVLink (CUDA IPC peer mapping): render and gather fused, a 4-byte all_reduce as completion barrier
    Device time (CUDA events on the launching stream) between barriers, max over ranks, best of 3."""
    w, h, nf, reps = 3840, 2160, 16, 3
    sh = stream.cuda_stream
    ctx.set_scene(*tpt.reference_scene(w, h))
    row0, nrows, rstep = mg.rows_of_rank(h, rank, world)

    def timed(fn, everyone=True):
        best = None
        for rep in range(reps + 1):                                # first repetition = warm-up
            torch.cuda.synchronize(dev); dist.barrier(); torch.cuda.synchronize(dev)
            e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            if everyone or rank == 0:
                fn()
            e1.record(stream)
            torch.cuda.synchronize(dev)
            t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            if rep > 0:
                best = t.item() if best is None else min(best, t.item())
        return best

    ctx.set_option("fast_variant", 3)
    full = torch.zeros((h, w, 4), dtype=torch.float32, device=dev) if rank == 0 else None
    ctx.read_ray_count(sh)
    one_ms = timed(lambda: ctx.draw(0, nf, w, h, full, flags=2, mode=tpt.MODE_FAST, stream=sh, want_rays=False), everyone=False)
    rays = mg.sum_ray_counts(ctx.read_ray_count(sh), dev) // (reps + 1)
    del full
    band = torch.zeros((nrows, w, 4), dtype=torch.float32, device=dev)
    out = [None]
    def method_a():
        ctx.draw(0, nf, w, h, band, flags=2, mode=tpt.MODE_FAST, rows=(row0, nrows, rstep, 1), stream=sh, want_rays=False)
        out[0] = mg.gather_rows(band, h, rank, world)
    a_ms = timed(method_a)
    rays_a = mg.sum_ray_counts(ctx.read_ray_count(sh), dev) // (reps + 1)
    img_a = out[0]
    ctx.set_option("fast_variant", 5)
    ctx.set_option("fast_alpha_zero", 1)                           # the peer image is write-only for the other ranks
    shared = mg.SharedImage(ctx, w, h, rank)
    done = torch.zeros(1, device=dev)
    def method_b():
        ctx.draw(0, nf, w, h, shared.ptr, flags=2, mode=tpt.MODE_FAST, rows=(row0, nrows, rstep, 0), stream=sh, want_rays=False)
        dist.all_reduce(done)
    b_ms = timed(method_b)
    rays_b = mg.sum_ray_counts(ctx.read_ray_count(sh), dev) // (reps + 1)
    rel = None
    if rank == 0:
        import numpy as _np
        b = shared.to_host()[..., :3].astype(_np.float64)
        a = img_a.cpu().numpy()[..., :3].astype(_np.float64)
        rel = float(_np.sqrt(((a - b) ** 2).sum() / (a ** 2).sum()))
    dist.barrier()
    shared.close()
    ctx.set_option("fast_variant", 3)
    ctx.set_option("fast_alpha_zero", 0)
    ctx.set_scene(*tpt.reference_scene(W, H))
    return {"workload": "46 spheres, 3840x2160, 64 spp (frames 0..15) — BASELINE configs[3]; rows interleaved over the ranks",
            "rays": rays, "one_gpu_ms": one_ms, "one_gpu_mray_s": rays / one_ms / 1e3,
            "A_nccl_allgather": {"ms": a_ms, "mray_s": rays_a / a_ms / 1e3, "speedup_vs_one_gpu": one_ms / a_ms, "kernel": "k_fast_queue"},
            "B_fused_peer_writeout": {"ms": b_ms, "mray_s": rays_b / b_ms / 1e3, "speedup_vs_one_gpu": one_ms / b_ms, "kernel": "k_fast_tileq"},
            "relL2_A_vs_B": rel, "timing": "CUDA events between barriers, max over ranks, best of 3 after one warm-up"}


if __name__ == "__main__":
    main()
