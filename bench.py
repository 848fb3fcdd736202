#!/usr/bin/env python
"""bench.py — geodesic rays/s and ms/frame of the 4K Schwarzschild lensed render.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (BASELINE.json metric "geodesic rays/sec and ms/frame at 4K"; SURVEY.md §8d):
the image_lens pipeline — per-pixel viewing angle (float32 table semantics) -> Binet RK4
null-geodesic trace (fp64, the reference's own RK4 stepper; hybrid arithmetic, see `arithmetic`
in config) -> deflection remap of a synthetic RGB checkerboard — at 3840x2160, M=1, r_obs=100 M,
vertical FOV 40 deg, psi=(0,0).  One step = one frame = ONE launch of the fused kernel
(lp_render_frame) per GPU.

Image format (all N, `value` and `e2e` alike): the 8-bit boundary of the reference's
image_lens.main — a uint8 RGB image in (imread; /255 -> float32, image_lens.py:448-450), the
float32 pipeline, an 8-bit frame out (imsave, :510) — LP_DTYPE_U8_UNIT: bytes in, bytes out,
/255 and trunc(255 v) on the device, pixel-identical to converting on the host.  The float32-RGB
variant of round 1 is reported beside it at N = 1 (`float32_frames`).

N > 1: weak scaling by rows — the frame grows to 3840 x (2160 N) at the same pixel scale, every
rank renders 2160 rows of it, interleaved in bands of 27 rows (the black hole sits in the centre
rows, so contiguous tiles are unevenly expensive), and every rank's kernel stores its pixels
straight into rank 0's frame over NVLink peer memory (dist.PeerFrame; --gather nccl: NCCL band
gather).  The same run also measures BASELINE config 4 (7680x4320 strong-scaled over the ranks,
against the same run's 1-rank time, gathered frame compared bit for bit with the 1-rank frame)
and config 5 (512 frames of 1024x1024, frame-sharded) — `config4_8k_strong`, `config5_sweep`.

Prints ONE JSON line on rank 0 (contract in the task statement): value = whole-job rays/s with
the source image resident in HBM; e2e = the same through the host-buffer API with the H2D copy of
the source and the D2H copy of the frame inside the timed region; roofline = the fused kernel's
algorithmic fp64 flops (43/RK4 step + 40/ray, SURVEY.md §8d) over its CUDA-event time against
the FP64 peak MEASURED in this run by a DFMA micro-benchmark (MEASURED_PEAKS.json has no fp64
figure; the nominal peak and the fraction of it are given too); cpu_baseline = the oracle (C/numpy
port of the reference's CPU path) timed on this box's host cores.

--impl reference times that CPU port alone (all host threads), one bounded sample per step.

--dump-outputs DIR (GPU arm, rank 0): after the timed steps, the frame the last timed step
returned, as a fixed seeded sample of its pixels (dump_frame), so that two builds run with the
same arguments can be compared pixel for pixel.
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

H0, W0 = 2160, 3840
M, R_OBS, VFOV_DEG = 1.0, 100.0, 40.0
FLOP_PER_STEP, FLOP_PER_RAY = 43, 40     # SURVEY.md §8d work model of the integrator
FP64_NOMINAL_TF = 148 * 64 * 2 * 1.965e9 / 1e12   # 148 SMs x 64 FMA/clk x 2 flop x 1.965 GHz
REF_SAMPLE_STRIDE = 8                    # CPU legs: every 8th row of the frame


def _oracle():
    """The CPU checker (oracle/), imported ONLY by the cpu_baseline leg and --impl reference."""
    p = os.path.join(ROOT, "oracle")
    if p not in sys.path:
        sys.path.insert(0, p)
    import lp_oracle
    return lp_oracle


def fov_for(H, W):
    """40 deg vertical FOV for the 2160-row frame; a taller (weak-scaled) frame keeps the same
    pixel scale, i.e. tan(vfov/2) grows with H, so every GPU's rows hold the same kind of rays as
    the single-GPU frame.  hfov from vfov as image_lens.py:461-463."""
    vfov = 2 * np.arctan(np.tan(np.radians(VFOV_DEG) / 2) * H / H0)
    return (2 * np.arctan(np.tan(vfov / 2) * W / H), vfov)


# ---------------------------------------------------------------------------------------
# clocks / throttle reasons during the timed region (NVML, sampled from a thread)
# ---------------------------------------------------------------------------------------
class ClockSampler:
    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nv = None

    def _run(self):
        nv = self.nv
        names = {"hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4),
                 "hw_power_brake": getattr(nv, "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80)}
        while not self._stop.is_set():
            try:
                self.samples.append(int(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                try:
                    mask = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                except Exception:
                    mask = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                for k, bit in names.items():
                    if mask & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.005)

    def __enter__(self):
        if self.nv is not None:
            self._thread = threading.Thread(target=self._run, daemon=True)
            self._thread.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self._thread is not None:
            self._thread.join()

    def summary(self):
        return {"sm_mhz": int(np.median(self.samples)) if self.samples else None,
                "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


# ---------------------------------------------------------------------------------------
# CPU legs (oracle port of the reference's numpy/numba path) — checker code, timed only
# ---------------------------------------------------------------------------------------
def cpu_frame(O, src8, H, W, rows=None):
    """image_lens.main's compute on the host (image_lens.py:448-510) for the frame rows `rows`
    (None = all): uint8 image -> float32/255 -> build_alpha_lookup -> precompute_final_alpha_lookup
    -> render_lensed_image -> 8-bit frame.  Returns (seconds, rays)."""
    fov = fov_for(H, W)
    t0 = time.perf_counter()
    img = src8.astype(np.float32) / 255.0
    alpha = O.build_alpha_lookup((H, W), fov, rows=rows)
    fa, w, n, _ = O.precompute_final_alpha_lookup(alpha, M, R_OBS)
    out = O.render_lensed_image(img, fa, w, fov, rows=rows)
    (np.clip(out, 0.0, 1.0) * 255).astype(np.uint8)
    return time.perf_counter() - t0, int(alpha.size)


def cpu_sample_text(W, H, rays, cores):
    return ("every %dth row of the %dx%d frame (%d rays) per step; trace on %d OpenMP threads, uint8 -> float32 "
            "conversion, alpha lookup, remap and the 8-bit conversion single-threaded numpy like the reference"
            % (REF_SAMPLE_STRIDE, W, H, rays, cores))


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # torchrun exports OMP_NUM_THREADS=1 to every rank; this arm is the only work on the box and
    # must use all the host threads it can, so size the OpenMP pool before libgomp initialises
    os.environ["OMP_NUM_THREADS"] = str(len(os.sched_getaffinity(0)))
    O = _oracle()
    O.build()
    from light_path_tracer_b200.synthetic import checkerboard
    H, W = H0 * args.gpus, W0
    src8 = checkerboard(H, W, np.uint8)
    rows = np.arange(0, H, REF_SAMPLE_STRIDE)              # bounded sample: every 8th row of the frame
    for _ in range(args.warmup):
        cpu_frame(O, src8, H, W, rows)
    times, rays = [], 0
    for _ in range(args.steps):
        t, rays = cpu_frame(O, src8, H, W, rows)
        times.append(t)
    total = float(np.sum(times))
    value = rays * args.steps / total
    cores = O.num_threads()
    line = {
        "impl": "reference", "metric": "geodesic rays/sec (4K Schwarzschild lensed render)",
        "value": value, "unit": "rays/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args.gpus, H, W, args.gather if args.gpus > 1 else "none"),
        "cpu_baseline": {"value": value, "unit": "rays/s", "cores": cores, "kind": "port",
                         "sample": cpu_sample_text(W, H, rays, cores)},
        "e2e": {"value": value, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def workload_config(n, H, W, gather_mode="peer", band_rows=None):
    if n > 1:
        how = ("every rank's render kernel stores its rows straight into rank 0's frame through NVLink peer "
               "memory (symmetric memory, 16-byte stores); completion = one 8-byte flag per rank (lp_peer_signal "
               "/ lp_peer_wait), no collective; two frame buffers" if gather_mode == "peer" else
               "each rank's rows rendered in bands whose NCCL gather to rank 0 overlaps the next band's render")
        par = "rows x%d: 2160 rows per GPU of a 3840x%d frame at the 1-GPU pixel scale, %s; %s" % (
            n, H, ("interleaved in bands of %d rows" % band_rows) if band_rows else "contiguous tiles", how)
    else:
        par = "single GPU"
    return {"workload": "image_lens Schwarzschild lensed render %dx%d (alpha lookup -> Binet RK4 trace -> remap), "
                        "M=1, r_obs=100M, vfov=40deg, psi=(0,0), synthetic RGB checkerboard through the 8-bit image "
                        "boundary of image_lens.main (uint8 image in, float32 pipeline semantics, 8-bit frame out)"
                        % (W, H),
            "rays_per_frame": H * W, "rows_per_gpu": H // n, "parallelism": par,
            "image_format": "uint8 RGB in / uint8 RGB out (LP_DTYPE_U8_UNIT); float32 frames beside it in "
                            "`float32_frames` (N = 1) / `weak_f32_frames` (N > 1)",
            "arithmetic": "hybrid (LP_TRACE_HYBRID, the image pipeline's default): FMA-contracted RK4 loop, strict "
                          "re-trace of the few rays that sweep more than 11.5 + ln max(final_alpha, 1e-3) rad inside r < 6M; same classification / winding / float32 "
                          "final_alpha as the strict kernel on this frame (tests/test_gpu_frame.py)",
            "l2": "256 MiB buffer written between timed steps (L2 flush)"}


def hbm_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs"
    except Exception:
        return 6650.0, "B200_PROFILING.md fallback (MEASURED_PEAKS.json absent)"


def ncu_traffic(kernel="lp_render_kernel"):
    """dram bytes per launch of a kernel from the committed ncu capture, if any (NOT measured in
    this run: `traffic_source` says so in the line)."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_summary.json")) as f:
            return json.load(f).get(kernel, {}).get("dram_bytes_per_launch")
    except Exception:
        return None


def ncu_executed(kernel="lp_render_kernel"):
    """Executed instructions per warp of a kernel (FP64-pipe / other) from the committed ncu source-level
    capture, if any: {"fp64": .., "other": .., "warps": .., "source": ..} or None."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_summary.json")) as f:
            e = json.load(f).get(kernel, {})
        if "fp64_inst_per_warp" in e:
            return {"fp64": float(e["fp64_inst_per_warp"]), "other": float(e["other_inst_per_warp"]),
                    "warps": float(e["warps"]), "source": e.get("source_page", e.get("source"))}
    except Exception:
        pass
    return None


TRAFFIC_SOURCE = "profiles/ncu_summary.json (committed ncu --set full capture of the same kernel; not re-measured in this run)"


def stat(ms):
    """mean / best / median of per-step times (ms)."""
    a = np.asarray(ms, dtype=np.float64)
    return {"mean": float(a.mean()), "best": float(a.min()), "median": float(np.median(a))}


DUMP_PIXELS = 1 << 21       # 2 M pixels: 24 MiB of float32 RGB + 16 MiB of float64 indices


def dump_frame(frame, out_dir):
    """Write a (H, W, C) frame tensor as out_dir/frame.npy: float32 (n, C), the pixels at the flat
    indices out_dir/frame_pixel_index.npy (float64, ascending), n = min(H W, DUMP_PIXELS) drawn
    without replacement from a generator with a fixed seed — the same pixels for every frame of
    that shape (a whole 4K frame in float32 would be 95 MiB)."""
    import torch
    n_px = frame.shape[0] * frame.shape[1]
    idx = np.sort(np.random.default_rng(0).choice(n_px, size=min(n_px, DUMP_PIXELS), replace=False))
    pix = frame.reshape(n_px, -1)[torch.from_numpy(idx).to(frame.device)].float().cpu().numpy()
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "frame.npy"), pix)
    np.save(os.path.join(out_dir, "frame_pixel_index.npy"), idx.astype(np.float64))


# ---------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------
def measure_fp64_peak(torch, ext):
    sink = torch.empty(148 * 32 * 256, dtype=torch.float64, device="cuda")
    iters, best = 20000, None
    for i in range(6):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        ext.bench_dfma(148 * 32, 256, iters, sink)
        b.record()
        torch.cuda.synchronize()
        ms = a.elapsed_time(b)
        if i and (best is None or ms < best):
            best = ms
    return 148 * 32 * 256 * iters * 16 / (best * 1e-3) / 1e12


def fp64_roofline(kernel, flops, kern_ms, peak_tf, traffic, flop_model, executed=None, sm_mhz=1965.0):
    achieved = flops / (kern_ms * 1e-3) / 1e12
    out = {"bound": "fp64", "kernel": kernel, "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s",
           "frac": achieved / peak_tf, "peak_nominal": FP64_NOMINAL_TF, "frac_of_nominal": achieved / FP64_NOMINAL_TF,
           "peak_source": "measured in this run: DFMA micro-benchmark lp_bench_dfma (MEASURED_PEAKS.json has no "
                          "fp64 entry); peak_nominal = 148 SM x 64 FMA/clk x 2 x 1.965 GHz",
           "flop_model": flop_model, "kernel_ms": kern_ms, "traffic": traffic, "traffic_source": TRAFFIC_SOURCE}
    if executed:
        # `achieved` counts the REFERENCE's operations (the algorithmic work SURVEY 8d defines); the kernel executes
        # fewer (FMA contraction, second-order form, scaled variable), so `frac` is work delivered per peak, not
        # pipe occupancy.  What the hardware did: executed instructions of the committed ncu source-level capture
        # (same kernel, same frame) over THIS run's kernel time.
        warps, f64, oth = executed["warps"], executed["fp64"], executed["other"]
        cycles = kern_ms * 1e-3 * sm_mhz * 1e6
        out["executed"] = {
            "fp64_inst_per_ray": f64, "other_inst_per_ray": oth,
            "fp64_pipe_frac": f64 * warps * 32 * 2 / (kern_ms * 1e-3) / 1e12 / peak_tf,
            "issue_port_frac": (2.0 * f64 + oth) * warps / (148 * 4) / cycles,
            "what": "fp64_pipe_frac = executed FP64 instructions x 2 flop / time / measured DFMA peak (FP64-pipe occupancy); "
                    "issue_port_frac = (2 x FP64 + other) warp instructions per SM sub-partition / elapsed cycles at "
                    "%d MHz (an FP64 instruction holds the dispatch port for two cycles): the rate this kernel runs at — an "
                    "empirical model, within a few per cent (ncu: issue active + FP64 pipe active / 2 = 101-104 %% of the "
                    "cycles; a value slightly above 1 means some instructions issued in the shadow of an FP64 one)" % sm_mhz,
            "source": "%s (instruction counts; not re-measured in this run)" % executed["source"]}
    return out


def run_gpu(args):
    import torch
    import torch.distributed as dist
    from light_path_tracer_b200 import _device as dev, _lib
    from light_path_tracer_b200 import image_lens as il
    from light_path_tracer_b200 import dist as lpdist
    from light_path_tracer_b200.metrics import Schwarzschild
    from light_path_tracer_b200.synthetic import checkerboard

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit("--gpus %d but WORLD_SIZE=%d: launch with torch.distributed.run" % (args.gpus, world))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    # one process per GPU: run on (and take pinned host memory from) the GPU's own NUMA node
    numa_node = dev.bind_to_gpu_numa_node(local) if world > 1 else None
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    ext = _lib.ext()
    N = world
    H, W = H0 * N, W0
    fov = fov_for(H, W)
    metric = Schwarzschild(M)
    HYB = dev.TRACE_HYBRID

    def barrier():
        if N > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if N == 1:
            return float(x)
        t = torch.tensor([float(x)], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0])

    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def timed(step, k, flush_l2=True):
        """k steps, each bracketed by CUDA events on the launching stream; L2 flushed in between.
        One untimed call first: the first launch of a kernel pays CUDA's lazy module load."""
        step()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(k)]
        barrier()
        for a, b in ev:
            if flush_l2:
                flush.zero_()
            a.record()
            step()
            b.record()
        barrier()
        return [a.elapsed_time(b) for a, b in ev]

    # ---- source images --------------------------------------------------------------------
    src8_np = checkerboard(H, W, np.uint8)
    src8_host = torch.from_numpy(src8_np).pin_memory()
    src8 = src8_host.to("cuda", non_blocking=True)

    # ---- where the rows go ------------------------------------------------------------------
    band_rows = lpdist.band_layout(H, N) if N > 1 else None
    gather_mode, pf, bg = "none", None, None
    if N > 1:
        gather_mode = args.gather
        if gather_mode == "peer":
            try:
                pf = lpdist.PeerFrame(H, (W, 3), torch.uint8, device, dst=0, band_rows=band_rows)
            except RuntimeError as exc:    # symmetric memory unavailable (agreed on by all ranks)
                sys.stderr.write("PeerFrame unavailable (%r): falling back to the NCCL band gather\n" % (exc,))
                gather_mode = "nccl"
        if gather_mode == "nccl":
            band_rows = None
            bg = lpdist.BandGather(H // N, (W, 3), torch.uint8, "cuda", dst=0, bands=args.bands)
    if band_rows:
        row0, rows, bands, frame_rows = lpdist.band_rows_of(H, rank, N, band_rows)
    else:
        row0, rows = lpdist.row_tiles(H, N)[rank]
        bands, frame_rows = None, np.arange(row0, row0 + rows)
    local_tile = torch.empty((rows, W, 3), dtype=torch.uint8, device="cuda")

    def render_local(out=local_tile, stats=None, src=src8, flags=HYB | dev.RENDER_STAGED_STORES, unit=True):
        il.render_frame(src, fov, R_OBS, metric, rows=(row0, rows), bands=bands, out=out, stats=stats, flags=flags,
                        unit_u8=unit)

    def step_resident():
        if pf is not None:
            tile, r, b, extra = pf.begin()
            il.render_frame(src8, fov, R_OBS, metric, rows=r, bands=b, out=tile, flags=HYB | extra, unit_u8=True)
            return pf.complete()
        if bg is None:
            render_local()
            return local_tile
        for first, n in bg.bands:
            il.render_frame(src8, fov, R_OBS, metric, rows=(row0 + first, n), out=bg.tile[first:first + n],
                            flags=HYB, unit_u8=True)
            bg.push(first, n)
        return bg.finish()

    # ---- work model numerator (sum of RK4 steps of this rank's rows) and the FP64 peak ----------
    stats = dev.new_stats()
    render_local(stats=stats)
    st = dev.read_stats(stats)
    flops_tile = FLOP_PER_STEP * st["sum_steps"] + FLOP_PER_RAY * st["n_rays"]
    peak_tf = measure_fp64_peak(torch, ext)

    # ---- value: device-resident steps ---------------------------------------------------------
    for _ in range(args.warmup):
        step_resident()
    last = [None]          # the frame the latest step returned (rank 0; None elsewhere)

    def step_kept():
        last[0] = step_resident()
    with ClockSampler(local) as clk:
        ms = timed(step_kept, args.steps)
    total_ms = max_over_ranks(float(np.sum(ms)))
    ms_stat = stat(ms)
    if args.dump_outputs and rank == 0:
        # before any later step can reuse the frame buffer (peer gather: two buffers, one more step)
        dump_frame(last[0], args.dump_outputs)

    # ---- N > 1: rank 0 re-renders the gathered frame alone, in row chunks, and compares -----------
    gather_identical = None
    if N > 1:
        frame = step_resident()
        torch.cuda.synchronize()
        if rank == 0:
            gather_identical = True
            chunk = 540
            for r0 in range(0, H, chunk):
                ref = il.render_frame(src8, fov, R_OBS, metric, rows=(r0, min(chunk, H - r0)), unit_u8=True)
                gather_identical = gather_identical and bool(torch.equal(ref, frame[r0:r0 + ref.shape[0]]))
        barrier()

    # ---- dominant kernel alone (no gather), same events: roofline numerator / denominator --------
    ms_k = timed(render_local, args.steps)
    kern_ms = max_over_ranks(float(np.mean(ms_k)))

    # ---- e2e: host buffers in and out every frame ---------------------------------------------
    # N = 1: image_lens.HostFramePipeline; N > 1: dist.ShardedHostFrames (every rank uploads its 1/N
    # of the rows of the NEW source over its own PCIe link, an NCCL all-gather over NVLink replicates
    # it; version=None = a new image every frame).  uint8 in, uint8 out.
    tile_hosts = [torch.empty((rows, W, 3), dtype=torch.uint8).pin_memory() for _ in range(3)]
    if N == 1:
        host_pipe = il.HostFramePipeline((H, W, 3), torch.uint8, VFOV_DEG, metric, depth=3, unit_u8=True)

        def submit(j, version=None):
            host_pipe.submit(src8_host, R_OBS, out=tile_hosts[j % 3], rows=(row0, rows), fov=fov,
                             flags=HYB | dev.RENDER_STAGED_STORES)
    else:
        host_pipe = lpdist.ShardedHostFrames((H, W, 3), torch.uint8, metric=metric, depth=3, unit_u8=True,
                                             band_rows=band_rows)

        def submit(j, version=None):
            host_pipe.submit(src8_host, fov, R_OBS, out=tile_hosts[j % 3], version=version,
                             flags=HYB | dev.RENDER_STAGED_STORES)

    def timed_e2e(k, version=None):
        for j in range(max(2, args.warmup)):
            submit(j, version)
        host_pipe.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        a.record()
        for j in range(k):
            submit(j, version)
        for slot in host_pipe._slots:
            torch.cuda.current_stream().wait_stream(slot["stream"])
        b.record()
        barrier()
        return max_over_ranks(a.elapsed_time(b))

    total_e2e = timed_e2e(args.steps)
    # the frame that came back through the host path is the frame the resident path renders
    render_local()
    if not torch.equal(tile_hosts[(args.steps - 1) % 3], local_tile.cpu()):
        raise SystemExit("e2e frame differs from the device-resident frame")

    # ---- the same bytes with no kernel: every rank's H2D and D2H copies alone, all ranks at once ----
    # (what the host side of the box can move; N GPUs share its PCIe root complex / DRAM)
    def copies_only(k, up=True):
        # the e2e leg's own traffic pattern without the kernel: three slots on three streams, slot j uploads
        # this rank's share of the pinned source (== its tile, in bytes) and then downloads the tile
        n_up = rows * W * 3
        h_in = src8_host.reshape(-1)[:n_up]
        d_ins = [torch.empty(n_up, dtype=torch.uint8, device="cuda") for _ in range(3)]
        d_out = local_tile.reshape(-1)
        streams = [torch.cuda.Stream() for _ in range(3)]

        def one(j):
            with torch.cuda.stream(streams[j % 3]):
                if up:
                    d_ins[j % 3].copy_(h_in, non_blocking=True)
                tile_hosts[j % 3].reshape(-1).copy_(d_out, non_blocking=True)
        for j in range(6):
            one(j)
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        a.record()
        for s_ in streams:
            s_.wait_stream(torch.cuda.current_stream())
        for j in range(k):
            one(j)
        for s_ in streams:
            torch.cuda.current_stream().wait_stream(s_)
        b.record()
        barrier()
        return max_over_ranks(a.elapsed_time(b))
    total_copies = copies_only(args.steps)
    total_copies_down = copies_only(args.steps, up=False)
    e2e_static = None
    if N > 1:
        # the same with an UNCHANGED background (parameter sweeps, BASELINE config 5): the source
        # stays resident, a step moves camera parameters in and the tile out
        total_static = timed_e2e(args.steps, version=1)
        e2e_static = {"value": H * W * args.steps / (total_static * 1e-3), "unit": "rays/s",
                      "ms_per_frame": total_static / args.steps,
                      "copies_only_ms_per_frame": total_copies_down / args.steps, "h2d_bytes_per_step": 0,
                      "d2h_bytes_per_step": int(H * W * 3),
                      "path": "dist.ShardedHostFrames with an unchanged source version: no upload, no all-gather"}

    extra = {}
    if N > 1:
        extra.update(multi_gpu_records(args, torch, dist, il, lpdist, dev, metric, rank, N, device, timed, barrier,
                                       max_over_ranks, checkerboard))
    if rank == 0 and N == 1:
        import contextlib
        with contextlib.redirect_stdout(sys.stderr):     # the reference-facing calls print progress lines
            extra.update(single_gpu_records(args, torch, il, dev, metric, ext, timed, src8_host, fov, H, W,
                                            flops_tile, peak_tf, checkerboard))

    # ---- sums over ranks ----------------------------------------------------------------------
    if N > 1:
        t = torch.tensor([float(flops_tile), float(st["sum_steps"]), float(st["sum_warp_steps"])],
                         dtype=torch.float64, device="cuda")
        tmax = t.clone()
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        flops_max_tile, sum_steps, sum_warp = float(tmax[0]), float(t[1]), float(t[2])
    else:
        flops_max_tile, sum_steps, sum_warp = float(flops_tile), float(st["sum_steps"]), float(st["sum_warp_steps"])

    if rank == 0:
        rays = H * W
        value = rays * args.steps / (total_ms * 1e-3)
        launches_per_step = len(bg.bands) if bg is not None else 1
        if pf is not None:
            launches_per_step += 2      # lp_peer_signal + lp_peer_wait (the root also releases: +1 there)
        line = {
            "metric": "geodesic rays/sec (4K Schwarzschild lensed render)",
            "value": value, "unit": "rays/s", "n_gpus": N, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": total_ms / args.steps, "ms_per_step_best": ms_stat["best"],
            "ms_per_step_median": ms_stat["median"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(N, H, W, gather_mode, band_rows),
            "ms_per_frame": total_ms / args.steps,
            "e2e": {"value": rays * args.steps / (total_e2e * 1e-3), "unit": "rays/s",
                    "ms_per_frame": total_e2e / args.steps,
                    "copies_only_ms_per_frame": total_copies / args.steps,
                    "copies_only_host_bytes_per_s": rays * 6 * args.steps / (total_copies * 1e-3),
                    "copies_only_what": "the same H2D + D2H copies of every rank on the same three-slot / three-stream "
                                        "pattern with no kernel in between, all ranks at once (max over ranks): the "
                                        "host-side floor of this box for the e2e leg",
                    "h2d_bytes_per_step": int(rays * 3), "d2h_bytes_per_step": int(rays * 3),
                    "path": ("image_lens.HostFramePipeline: pinned uint8 source -> H2D -> lp_render_frame -> D2H "
                             "pinned uint8 frame, every frame; 3 slots on 3 streams")
                    if N == 1 else
                            ("dist.ShardedHostFrames: every frame is a NEW pinned uint8 source — every rank uploads "
                             "its 1/N of the rows, NCCL all-gather replicates it over NVLink, lp_render_frame renders "
                             "the rank's rows, D2H of the rows to pinned memory; 3 slots on 3 streams")},
            "host": {"numa_node_of_rank0": numa_node, "cpus_rank0": len(os.sched_getaffinity(0)),
                     "e2e_host_bytes_per_s": rays * 6 * args.steps / (total_e2e * 1e-3),
                     "note": "every rank is pinned to its GPU's NUMA node before it allocates pinned memory "
                             "(_device.bind_to_gpu_numa_node); e2e_host_bytes_per_s = host->device + device->host "
                             "bytes of all ranks per second of the e2e leg"},
            "gpu_launches": args.steps * launches_per_step,
            "gather": gather_mode,
            "roofline": fp64_roofline("lp_render_kernel (alpha + Binet RK4 + remap, fused)", flops_max_tile, kern_ms,
                                      peak_tf, ncu_traffic(),
                                      "43 flop per RK4 step + 40 per ray (SURVEY.md 8d), the reference's own operation "
                                      "count; the hybrid loop issues 14 FP64 instructions per step (second-order form of "
                                      "the same RK4 step in the scaled variable 3Mu; strict: 34, ceiling 0.5 by construction), "
                                      "so `frac` is the reference's work delivered per peak, not pipe occupancy.  The kernel is bound by "
                                      "the SM sub-partition's issue port: an FP64 instruction holds it for 2 cycles, any "
                                      "other for 1, and 2 x FP64 + other instructions = the elapsed cycles (`executed`)",
                                      executed=ncu_executed() if N == 1 else None,
                                      sm_mhz=float((clk.summary() or {}).get("sm_mhz") or 1965.0)),
            "kernel_ms_per_step": stat(ms_k),
            "rk4_steps_per_frame": sum_steps,
            "lane_efficiency": sum_steps / sum_warp if sum_warp else None,
            "clocks": clk.summary(),
        }
        if gather_identical is not None:
            line["gather_bit_identical"] = gather_identical
        if e2e_static is not None:
            line["e2e_static_source"] = e2e_static
        line.update(extra)
        if N == 1 and not args.no_cpu:
            cpu_legs(line, il, src8_np, fov, H, W)
        print(json.dumps(line), flush=True)
    if pf is not None:
        pf.drain()
    if N > 1:
        dist.destroy_process_group()


def multi_gpu_records(args, torch, dist, il, lpdist, dev, metric, rank, N, device, timed, barrier, max_over_ranks,
                      checkerboard):
    """N > 1: the weak frame with float32 pixels, BASELINE config 4 (8K strong) and config 5 (sweep)."""
    HYB = dev.TRACE_HYBRID
    out = {}
    reps = max(5, min(args.steps, 20))

    def peer_step(pf, src, fov, unit):
        def step():
            tile, r, b, extra = pf.begin()
            il.render_frame(src, fov, R_OBS, metric, rows=r, bands=b, out=tile, flags=HYB | extra, unit_u8=unit)
            return pf.complete()
        return step

    # ---- the weak frame with float32 RGB pixels (round 1's format): 4x the NVLink bytes -----------
    H, W = H0 * N, W0
    fov = fov_for(H, W)
    try:
        src32 = torch.from_numpy(checkerboard(H, W, np.float32)).cuda()
        pf32 = lpdist.PeerFrame(H, (W, 3), torch.float32, device, dst=0, band_rows=lpdist.band_layout(H, N))
        ms = max_over_ranks(float(np.mean(timed(peer_step(pf32, src32, fov, False), reps))))
        out["weak_f32_frames"] = {"ms_per_step": ms, "value": H * W / ms * 1e3, "unit": "rays/s",
                                  "nvlink_bytes_into_rank0_per_step": int((N - 1) * (H // N) * W * 12),
                                  "what": "the same weak-scaled frame with float32 RGB source and frame (12 B/pixel "
                                          "over NVLink instead of 3)"}
        pf32.drain()
        del pf32, src32
    except RuntimeError as exc:
        out["weak_f32_frames"] = {"error": repr(exc)[:200]}
    torch.cuda.empty_cache()

    # ---- config 4: 7680x4320, strong scaling over the ranks, frame assembled on rank 0 -------------
    H4, W4 = 4320, 7680
    fov4 = fov_for(H0, W0)                       # 40 deg vertical, 16:9 (same aspect as the 4K frame)
    src4 = torch.from_numpy(checkerboard(H4, W4, np.uint8)).cuda()
    rec = {"frame": "%dx%d" % (W4, H4), "rays": H4 * W4, "image_format": "uint8 in / uint8 out (LP_DTYPE_U8_UNIT)"}
    full = None
    if rank == 0:
        full = torch.empty((H4, W4, 3), dtype=torch.uint8, device="cuda")
    # the same run's 1-rank time: rank 0 renders the whole frame alone (the others wait)
    if rank == 0:
        def single():
            il.render_frame(src4, fov4, R_OBS, metric, out=full, unit_u8=True, flags=HYB | dev.RENDER_STAGED_STORES)
        t1 = float(np.mean(timed_local(torch, single, 5)))
    else:
        t1 = 0.0
    barrier()
    t1 = max_over_ranks(t1)
    rec["ms_1_rank"] = t1
    b4 = lpdist.band_layout(H4, N)
    try:
        pf4 = lpdist.PeerFrame(H4, (W4, 3), torch.uint8, device, dst=0, band_rows=b4)
        step4 = peer_step(pf4, src4, fov4, True)
        ms = max_over_ranks(float(np.mean(timed(step4, reps))))
        got = step4()
        torch.cuda.synchronize()
        same = bool(torch.equal(got, full)) if rank == 0 else None
        barrier()
        rec["peer"] = {"ms_per_frame": ms, "rays_per_s": H4 * W4 / ms * 1e3, "speedup_vs_1_rank": t1 / ms,
                       "band_rows": b4, "gather_bit_identical": same, "timed_out": pf4.timed_out(),
                       "how": "rows interleaved in bands, stored into rank 0's frame over NVLink by the render "
                              "kernels (dist.PeerFrame), flags for completion"}
        pf4.drain()
        del pf4
    except RuntimeError as exc:
        rec["peer"] = {"error": repr(exc)[:200]}
    # NCCL variant: contiguous tiles rendered in bands, each band gathered while the next renders
    rs = lpdist.RowShardedRenderer(src4, VFOV_DEG, metric)
    g4 = lpdist.BandGather(H4 // N, (W4, 3), torch.uint8, "cuda", dst=0, bands=args.bands)

    def nccl_step():
        r0, _ = rs.tiles[rank]
        for first, n in g4.bands:
            il.render_frame(src4, fov4, R_OBS, metric, rows=(r0 + first, n), out=g4.tile[first:first + n],
                            flags=HYB, unit_u8=True)
            g4.push(first, n)
        return g4.finish()
    ms = max_over_ranks(float(np.mean(timed(nccl_step, reps))))
    got = nccl_step()
    torch.cuda.synchronize()
    same = bool(torch.equal(got, full)) if rank == 0 else None
    rec["nccl"] = {"ms_per_frame": ms, "rays_per_s": H4 * W4 / ms * 1e3, "speedup_vs_1_rank": t1 / ms,
                   "gather_bit_identical": same,
                   "how": "contiguous tiles in %d bands, NCCL gather of each band overlapped with the next band's "
                          "render (dist.BandGather)" % args.bands}
    out["config4_8k_strong"] = rec
    del rs, g4, src4, full
    torch.cuda.empty_cache()

    # ---- config 5: 512 frames of 1024x1024, frame-sharded, no data-path collective -----------------
    Hs = Ws = 1024
    src5 = torch.from_numpy(checkerboard(Hs, Ws, np.uint8)).cuda()
    pipe = il.LensPipeline(src5, VFOV_DEG, metric)
    grid = lpdist.sweep_grid()
    mine = lpdist.frame_shard(len(grid), rank, N)
    frames = torch.empty((len(mine), Hs, Ws, 3), dtype=torch.uint8, device="cuda")

    def sweep():
        for j, k in enumerate(mine):
            r_obs, psi = grid[k]
            pipe.render(r_obs, psi=psi, out=frames[j], unit_u8=True)
    ms_plain = max_over_ranks(float(np.mean(timed(sweep, 2, flush_l2=False))))
    check = frames[-1].clone()
    graph = pipe.capture_sweep([grid[k] for k in mine], frames, unit_u8=True)
    ms_graph = max_over_ranks(float(np.mean(timed(graph.replay, 2, flush_l2=False))))
    same = bool(torch.equal(check, frames[-1]))
    out["config5_sweep"] = {"frames": len(grid), "frame": "1024x1024", "frames_per_rank": len(mine),
                            "ms_total": ms_plain, "ms_total_cuda_graph": ms_graph,
                            "rays_per_s": len(grid) * Hs * Ws / min(ms_plain, ms_graph) * 1e3,
                            "graph_same_frames": same,
                            "grid": "32 r_obs in geomspace(15, 1000) x 16 pitches in linspace(-15, 15) deg, "
                                    "round-robin over the ranks; schedule (re-packing or not) chosen per frame"}
    return out


def timed_local(torch, fn, k):
    """Events on this rank only (no barrier): used while the other ranks idle."""
    fn()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(k)]
    for a, b in ev:
        a.record()
        fn()
        b.record()
    torch.cuda.synchronize()
    return [a.elapsed_time(b) for a, b in ev]


def single_gpu_records(args, torch, il, dev, metric, ext, timed, src8_host, fov, H, W, flops_tile, peak_tf,
                       checkerboard):
    """N = 1: the other kernels and BASELINE configs that fit one GPU, the float32-frame variant,
    and the drop-in (numpy in / numpy out) end-to-end time."""
    HYB = dev.TRACE_HYBRID
    hbm, hbm_src = hbm_peak()
    rays = H * W
    mean = lambda fn: float(np.mean(timed(fn, args.steps)))      # noqa: E731
    src32_np = checkerboard(H, W, np.float32)
    src32_host = torch.from_numpy(src32_np).pin_memory()
    src32 = src32_host.cuda()
    tile32 = torch.empty((H, W, 3), dtype=torch.float32, device="cuda")
    a32 = il.build_alpha_lookup((H, W), fov, device=True)
    fa32, w16 = metric.trace_alpha_table(a32, R_OBS)

    def tf(ms):
        # tflops: the REFERENCE's operation count (43 flop / RK4 step + 40 / ray) per second.  The FMA loop executes
        # 14 FP64 instructions per step for those 43 flops, so this ratio is work delivered per peak and can pass 1.
        return {"ms": ms, "rays_per_s": rays / ms * 1e3, "tflops": flops_tile / ms / 1e9,
                "frac_of_measured_fp64_peak": flops_tile / ms / 1e9 / peak_tf}

    t_f32 = mean(lambda: il.render_frame(src32, fov, R_OBS, metric, out=tile32))
    t_render_strict = mean(lambda: il.render_frame(src32, fov, R_OBS, metric, out=tile32, flags=0))
    t_repack = mean(lambda: il.render_frame(src32, fov, R_OBS, metric, out=tile32, flags=HYB | dev.TRACE_REPACK))
    t_strict = mean(lambda: metric.trace_alpha_table(a32, R_OBS, flags=0))
    t_fused = mean(lambda: metric.trace_alpha_table(a32, R_OBS, flags=1))
    t_hybrid = mean(lambda: metric.trace_alpha_table(a32, R_OBS, flags=4))
    t_remap = mean(lambda: il.render_lensed_image(src32, a32, fa32, w16, 0.0, fov))
    t_alpha = mean(lambda: il.build_alpha_lookup((H, W), fov, device=True))

    # float32 frames end to end (round 1's e2e): PCIe-bound, 2 x 99.5 MB per frame
    pipe32 = il.HostFramePipeline((H, W, 3), torch.float32, VFOV_DEG, metric, depth=3)
    out32 = [torch.empty((H, W, 3), dtype=torch.float32).pin_memory() for _ in range(3)]
    for j in range(3):
        pipe32.submit(src32_host, R_OBS, out=out32[j % 3], fov=fov)
    pipe32.synchronize()
    ea, eb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ea.record()
    for j in range(args.steps):
        pipe32.submit(src32_host, R_OBS, out=out32[j % 3], fov=fov)
    for slot in pipe32._slots:
        torch.cuda.current_stream().wait_stream(slot["stream"])
    eb.record()
    torch.cuda.synchronize()
    t_e2e32 = ea.elapsed_time(eb) / args.steps
    del pipe32, out32

    # ---- the drop-in path: the three reference-facing calls with numpy in / numpy out, exactly as
    # image_lens.main issues them (image_lens.py:480-505), wall clock ------------------------------
    def dropin(img, unit):
        t0 = time.perf_counter()
        alpha = il.build_alpha_lookup((H, W), fov)
        fa, w, n, _ = il.precompute_final_alpha_lookup(alpha, metric.alpha_crit(R_OBS), R_OBS, metric)
        frame = il.render_lensed_image(img, alpha, fa, w, metric.alpha_crit(R_OBS), fov, False, unit_u8=unit)
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) * 1e3, frame
    src8_np = src8_host.numpy()
    walls32, walls8 = [], []
    for j in range(7):
        ms32, fr32 = dropin(src32_np, False)
        ms8, fr8 = dropin(src8_np, True)
        if j >= 2:
            walls32.append(ms32)
            walls8.append(ms8)
    il.render_frame(src32, fov, R_OBS, metric, out=tile32)
    dropin_same = bool(np.array_equal(fr32, tile32.cpu().numpy()))
    # pinned PCIe rate of this box (one 99.5 MB copy each way, best of 5) for the floor
    h = torch.empty(rays * 12, dtype=torch.uint8).pin_memory()
    d = torch.empty(rays * 12, dtype=torch.uint8, device="cuda")
    best = [1e9, 1e9]
    for _ in range(5):
        for k, (dst, src) in enumerate(((d, h), (h, d))):
            ea, eb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ea.record()
            dst.copy_(src, non_blocking=True)
            eb.record()
            torch.cuda.synchronize()
            best[k] = min(best[k], ea.elapsed_time(eb))
    h2d_gbs, d2h_gbs = rays * 12 / best[0] / 1e6, rays * 12 / best[1] / 1e6
    del h, d
    up32, down32 = rays * (4 + 12 + 4 + 2), rays * (4 + 4 + 2 + 12)
    up8, down8 = rays * (4 + 3 + 4 + 2), rays * (4 + 4 + 2 + 3)
    floor32 = up32 / h2d_gbs / 1e6 + down32 / d2h_gbs / 1e6
    floor8 = up8 / h2d_gbs / 1e6 + down8 / d2h_gbs / 1e6
    e2e_dropin = {
        "what": "wall time per frame of build_alpha_lookup -> precompute_final_alpha_lookup -> "
                "render_lensed_image with numpy arrays in and out (image_lens.py:480-505), synchronous",
        "float32_image": {"ms_per_frame_best": float(np.min(walls32)), "ms_per_frame_median": float(np.median(walls32)),
                          "rays_per_s": rays / float(np.median(walls32)) * 1e3,
                          "h2d_bytes": int(up32), "d2h_bytes": int(down32), "pcie_floor_ms": floor32,
                          "ratio_to_floor": float(np.median(walls32)) / floor32,
                          "frame_equals_fused_kernel": dropin_same},
        "uint8_image_main_equivalent": {"ms_per_frame_best": float(np.min(walls8)),
                                        "ms_per_frame_median": float(np.median(walls8)),
                                        "rays_per_s": rays / float(np.median(walls8)) * 1e3,
                                        "h2d_bytes": int(up8), "d2h_bytes": int(down8), "pcie_floor_ms": floor8,
                                        "ratio_to_floor": float(np.median(walls8)) / floor8},
        "pcie_pinned_gbs": {"h2d": h2d_gbs, "d2h": d2h_gbs},
        "staging": "results land in pinned memory the returned numpy arrays own; pinned inputs (the tables this "
                   "package returned) upload in place; the pageable source image is staged in 8 MB chunks by a "
                   "thread pool while earlier chunks are on the link (_device.py)"}

    # ---- config 3 (generic 8-D RK45 integrator over the 4K alpha table) and a Kerr 4K lookup -------
    from light_path_tracer_b200 import geodesic_tracer as gt
    from light_path_tracer_b200.metrics import Kerr
    a64 = a32.double()

    def once(fn):
        fn()
        ea, eb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ea.record()
        res = fn()
        eb.record()
        torch.cuda.synchronize()
        return ea.elapsed_time(eb), res
    t_rk45, rk = once(lambda: gt.trace_rays(metric, R_OBS, a64))
    rk_attempts = float(((rk[3][..., 1].double() - 2) / 6).sum())
    kerr = Kerr(M, 0.9)
    cam_k = dev.camera_vector((H, W), fov, (0.0, 0.0), il._psi_frame)
    steps_k = torch.empty((H, W, 2), dtype=torch.int32, device="cuda")
    t_kerr, _ = once(lambda: kerr.trace_alpha_table_2d(a32, cam_k, R_OBS, np.pi / 2))
    kerr.trace_alpha_table_2d(a32, cam_k, R_OBS, np.pi / 2, steps=steps_k)
    kerr_attempts = float(steps_k[..., 1].double().sum())
    try:
        t_kerr_api, _ = once(lambda: il.precompute_final_alpha_lookup_2d(
            a32, fov, kerr.alpha_crit(R_OBS), R_OBS, kerr, theta_obs=np.pi / 2, psi=(0.0, 0.0)))
    except Exception as exc:                      # auxiliary figure only
        t_kerr_api = None
        sys.stderr.write("kerr API lookup skipped: %r\n" % (exc,))
    # flop models of the two adaptive integrators, recounted from the kernels as written
    # (DESIGN.md §4): FP64-pipe instructions per step attempt x 2 flop (every DFMA/DMUL/DADD slot
    # counted as one FMA = 2 flop, i.e. the fraction is the pipe-slot utilisation an ideal
    # schedule of the SAME instruction stream would reach)
    rk_slots, kerr_slots = RK45_FP64_SLOTS_PER_ATTEMPT, KERR_FP64_SLOTS_PER_ATTEMPT
    rk_tf = rk_attempts * rk_slots * 2 / t_rk45 / 1e9
    kerr_tf = kerr_attempts * kerr_slots * 2 / t_kerr / 1e9
    return {
        "float32_frames": {"value": rays / t_f32 * 1e3, "unit": "rays/s", "ms_per_step": t_f32,
                           "frac_of_measured_fp64_peak": flops_tile / t_f32 / 1e9 / peak_tf,
                           "e2e": {"value": rays / t_e2e32 * 1e3, "ms_per_frame": t_e2e32,
                                   "h2d_bytes_per_step": int(rays * 12), "d2h_bytes_per_step": int(rays * 12)},
                           "what": "the same frame with a float32 RGB source and frame (round 1's format)"},
        "e2e_dropin": e2e_dropin,
        "config3_rk45_frame_4k": {"ms": t_rk45, "rays_per_s": rays / t_rk45 * 1e3,
                                  "step_attempts_per_s": rk_attempts / t_rk45 * 1e3,
                                  "what": "geodesic_tracer.trace_ray semantics (scipy RK45, rtol 1e-8) for every "
                                          "pixel of the 3840x2160 alpha table, lp_rk45_eq_kernel (equatorial observer: four moving components)"},
        "roofline_rk45": {"bound": "fp64", "kernel": "lp_rk45_eq_kernel", "achieved": rk_tf, "peak": peak_tf,
                          "unit": "TFLOP/s", "frac": rk_tf / peak_tf, "frac_of_nominal": rk_tf / FP64_NOMINAL_TF,
                          "kernel_ms": t_rk45, "step_attempts": rk_attempts,
                          "flop_model": "%d FP64 instructions per step attempt and ray as executed by the equatorial "
                                        "four-component kernel (ncu recount, see RK45_FP64_SLOTS_PER_ATTEMPT in bench.py: 6 RHS "
                                        "evaluations, stage / error sums, controller) x 2 flop; the eight-component kernel "
                                        "executed 620, SURVEY 8d's estimate was ~750 flop per attempt" % rk_slots,
                          "traffic": ncu_traffic("lp_rk45_eq_kernel"), "traffic_source": TRAFFIC_SOURCE},
        "kerr_lookup_4k": {"ms": t_kerr, "rays_per_s": rays / t_kerr * 1e3, "ms_api_with_mirror": t_kerr_api,
                           "what": "Kerr a=0.9 M, equatorial observer: (alpha, theta) lookup of the full 3840x2160 "
                                   "frame without the top/bottom mirror, lp_kerr_queued_kernel; ms_api_with_mirror = "
                                   "image_lens.precompute_final_alpha_lookup_2d on the same device-resident alpha "
                                   "table (top half traced, bottom mirrored)"},
        "roofline_kerr": {"bound": "fp64", "kernel": "lp_kerr_queued_kernel", "achieved": kerr_tf, "peak": peak_tf,
                          "unit": "TFLOP/s", "frac": kerr_tf / peak_tf, "frac_of_nominal": kerr_tf / FP64_NOMINAL_TF,
                          "kernel_ms": t_kerr, "step_attempts": kerr_attempts,
                          "flop_model": "%d FP64-pipe instructions per step attempt as compiled (7 RHS evaluations of "
                                        "204 slots + stage / error sums) x 2 flop" % kerr_slots,
                          "traffic": ncu_traffic("lp_kerr_queued_kernel"), "traffic_source": TRAFFIC_SOURCE},
        "trace_kernel_strict": tf(t_strict), "trace_kernel_hybrid": tf(t_hybrid),
        "trace_kernel_fma_contracted": tf(t_fused),
        "render_kernel_strict": tf(t_render_strict),
        "render_kernel_repack_forced": dict(tf(t_repack), what="the same float32 frame through the lane re-packing "
                                            "schedule (LP_TRACE_REPACK); the default picks one ray per thread here"),
        "alpha_lookup_kernel": {"ms": t_alpha},
        "remap_kernel": {"ms": t_remap, "gb_per_s": rays * 30 / t_remap / 1e6, "bytes_per_px": 30,
                         "frac_of_measured_hbm": rays * 30 / t_remap / 1e6 / hbm},
        "roofline_remap": {"bound": "hbm", "kernel": "stand-alone remap of render_lensed_image (float32 RGB)",
                           "achieved": rays * 30 / t_remap / 1e6, "peak": hbm, "unit": "GB/s",
                           "frac": rays * 30 / t_remap / 1e6 / hbm,
                           "traffic": ncu_traffic("lp_remap_f32rgb_x4_kernel"), "traffic_source": TRAFFIC_SOURCE,
                           "peak_source": hbm_src},
    }


# FP64-pipe instructions per step attempt (per ray) of the two adaptive integrators as executed:
#   RK45 — the equatorial four-component kernel lp_rk45_eq_kernel: ncu source counts (profiles/r2ab_ncu_rk45.md,
#          960x540 rays, 293.4 attempts per ray): 667 330 FP64 warp instructions per warp x 2 368 warps x 27.8
#          active threads / 1.521e8 attempts = 289 (before the controller / right-hand-side trims of this round:
#          372; the eight-component kernel it replaced: 620);
#   Kerr — 7 right-hand sides of 204 FP64 instructions + 370 of stage / error sums, from the SASS (DESIGN.md §4).
RK45_FP64_SLOTS_PER_ATTEMPT = 289
KERR_FP64_SLOTS_PER_ATTEMPT = 1600


def cpu_legs(line, il, src8_np, fov, H, W):
    """cpu_baseline (rank 0, N = 1): the oracle port on the box's host cores, on the SAME bounded
    sample --impl reference times (every 8th row), plus CPU figures beside the two secondary kernels."""
    O = _oracle()
    O.build()
    rows = np.arange(0, H, REF_SAMPLE_STRIDE)
    cpu_frame(O, src8_np, H, W, rows)
    ts = []
    for _ in range(3):
        t_cpu, n_cpu = cpu_frame(O, src8_np, H, W, rows)
        ts.append(t_cpu)
    cores = O.num_threads()
    line["cpu_baseline"] = {"value": n_cpu / float(np.mean(ts)), "unit": "rays/s", "cores": cores, "kind": "port",
                            "sample": cpu_sample_text(W, H, n_cpu, cores) + " (3 steps after one warm-up; "
                                      "--impl reference times the same sample)"}
    stride = (H * W) // 32768
    a_s = O.build_alpha_lookup((H, W), fov).reshape(-1)[::stride].astype(np.float64)
    t0 = time.perf_counter()
    O.rk45_trace_batch(M, R_OBS, a_s)
    t_rk_cpu = time.perf_counter() - t0
    th_s = il._theta_pixel((H, W), fov, (0.0, 0.0), H).reshape(-1)[::stride]
    if "config3_rk45_frame_4k" in line:
        line["config3_rk45_frame_4k"]["cpu_port"] = {
            "rays_per_s": a_s.size / t_rk_cpu, "cores": cores,
            "sample": "every %dth pixel (%d rays), C port of scipy RK45 + events" % (stride, a_s.size)}
    if "kerr_lookup_4k" in line:
        t0 = time.perf_counter()
        O.kerr_trace_rays_batch(M, 0.9, R_OBS, a_s, np.asarray(th_s, np.float64), np.pi / 2)
        t_k_cpu = time.perf_counter() - t0
        line["kerr_lookup_4k"]["cpu_port"] = {
            "rays_per_s": a_s.size / t_k_cpu, "cores": cores,
            "sample": "every %dth pixel (%d rays), C restatement of the numba Kerr DP45 tracer" % (stride, a_s.size)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--bands", type=int, default=4, help="N > 1, NCCL band gather: bands per tile")
    ap.add_argument("--gather", default="peer", choices=["peer", "nccl"],
                    help="N > 1: peer = rows stored straight into rank 0's frame over NVLink peer memory; "
                         "nccl = NCCL gather of row bands overlapped with the render")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="GPU arm: write a seeded sample of the frame the last timed step returned to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
