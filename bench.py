#!/usr/bin/env python3
"""bench.py -- the driver's measurement contract for the svt-av1-psy B200 DSP tier.

  python bench.py --gpus N --steps K --warmup W                 B200 arm (libsvtav1_b200.so, T2 entry points)
  python bench.py --impl reference --gpus N --steps K --warmup W  reference arm: the reference's own kernels
                                                                (oracle/_ref, AVX2 intrinsics tier where it
                                                                builds without NASM, else C) on all host cores

A "step" = the hot-path DSP work of ONE 1920x1080 8-bit 4:2:0 frame at preset-8 / CRF-30 settings
(svt-av1-psy_b200/workload.py): open-loop ME (HME pyramid + 85-PU full-pel search, 2 references),
residual + forward transform + quantize + inverse/reconstruction of every sample, CDEF search + apply,
Wiener statistics + filter.  Prints ONE JSON line (rank 0).

`value`  : frames/s with every input already resident in HBM (CUDA events on the launch stream).
`e2e`    : same metric through the host-buffer path: per step the source picture and the prediction are copied
           from pinned host memory (the residual is formed on the device) and the ME results, per-block eobs +
           eob-bounded scan-order levels, CDEF costs and Wiener statistics are read back, inside the timed region
           (the restored picture stays on the device: it is the reference picture of later frames).
Each timed region is exactly --steps steps.  --dump-outputs DIR writes what the last timed step computed (dump_outputs).
"""
import argparse
import ctypes as ct
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the tree may be read-only: nothing is written there

# BASELINE.json's metric, verbatim.  What is timed under that name is the tier's hot path only (SURVEY.md 8): one
# "frame" = ME + transform/quantise/inverse + CDEF + Wiener work of one 1080p preset-8 picture, NOT a full encode --
# `metric_scope` in the JSON line and config.workload say so, for both arms.
METRIC = "1080p preset-8 encoded frames/sec at 1/2/4/8 B200 vs reference AVX2 on host"
METRIC_SCOPE = "hot path only (SURVEY 8: ME + transform/quant/inverse + CDEF + Wiener of one 1080p preset-8 frame per step), not a full encode"
N_FRAME_SETS = 8  # rotated between steps: no step finds its inputs in L2, and (e2e) up to 8 frames are in flight
N_CALLS = 10      # len(FramePipeline.CALLS): the T2 entry points one frame goes through
EXCH_BATCH = 4    # pictures per reconstructed-reference exchange (one mini-GOP slice per NCCL group launch)
# roofline.traffic: dram__bytes_read.sum + dram__bytes_write.sum of the dominant call's kernels, per launch, read from the committed ncu launch
# list of tools/profile_step.py for the same configuration (profiles/README.md) -- None when no capture of that configuration is committed
NCU_LAUNCHES = {1: "profiles/r2_launches_config1.csv", 2: "profiles/r2_launches_config2.csv"}
CALL_KERNELS = {"me_pyramid": ("downsample_2d_kernel", "pad_plane_kernel"), "me_search": ("me_b64_hme_kernel", "fullpel_search_kernel", "me_b64_finish_kernel"),
                "txfm_trio": ("trio_txfm_kernel",), "pack_levels": ("eob_chunk_sum_kernel", "eob_offsets_kernel", "pack_levels_kernel"),
                "cdef_search": ("cdef_dir_kernel", "cdef_search_kernel"), "cdef_apply": ("cdef_apply_kernel",),
                "lr_boundaries": ("lr_save_boundary_kernel",), "rest_extend": ("pad_planes_kernel",),
                "wiener_stats": ("stats_sum_kernel", "stats_mma_kernel", "stats_finalize_kernel", "stats_lag_"), "wiener_filter": ("lr_filter_kernel",)}


def ncu_dram_bytes(config, call):
    import csv
    path = os.path.join(ROOT, NCU_LAUNCHES.get(config, ""))
    if not os.path.isfile(path):
        return None, None
    tot, seen = 0.0, False
    for r in csv.reader(open(path)):
        if len(r) > 10 and r[0].isdigit() and r[-3].startswith("dram__bytes_") and any(k in r[4] for k in CALL_KERNELS.get(call, ())):
            tot += float(r[-1].replace(",", "")) * {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}.get(r[-2], 1.0)
            seen = True
    return (int(tot), NCU_LAUNCHES[config]) if seen else (None, None)


# ------------------------------------------------------------------------------------------------------
# reference arm: the reference's own kernels over the same work lists (oracle/ref_driver.c), whole frames
# in flight on a persistent core-pinned thread pool.  Imports NOTHING from the product package.
# ------------------------------------------------------------------------------------------------------
REF_TIER_NAME = {0: "c", 1: "avx2-intrinsics (inverse transform: the reference's intrinsics AVX2/SSE4.1 kernels; the dav1d NASM kernels cannot be assembled here)"}


def load_reference():
    import oracle
    if oracle.ref is None:
        return None, 0
    tier = oracle.ref.ref_set_tier(1)
    return oracle.ref, (1 if tier == 1 else 0)


def make_workloads(args, rank, n_sets):
    """the frame sets of this rank: same work lists, different synthetic content"""
    from oracle.frame_ref import load_workload_module
    W = load_workload_module()
    w, h, bd, preset = W.CONFIGS[args.config]
    if args.width:
        w, h = args.width, args.height
    wl0 = W.FrameWorkload(w, h, seed=20260923 + 17 * rank * N_FRAME_SETS, bit_depth=bd, preset=preset)
    return W, [wl0 if i == 0 else wl0.with_seed(20260923 + 17 * (rank * N_FRAME_SETS + i)) for i in range(n_sets)]


def host_threads():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def time_reference_frames(ref, frames, n_frames, n_threads, warm_frames):
    from oracle.frame_ref import run_frames
    run_frames(ref, frames, max(warm_frames, n_threads), n_threads)  # every worker touches its private buffers once
    return run_frames(ref, frames, n_frames, n_threads)


def reference_arm(args, wls, steps, warmup, budget_s=60.0):
    """-> dict(fps, ms, cores, tier, inner_repeats, scaling) or None.  A step = one whole frame; `steps` frames form a
    batch and the batch is repeated back to back (one continuous stream of frames, no barrier between repeats) so
    that every host thread has several frames to work through."""
    from oracle.frame_ref import RefFrame
    ref, tier = load_reference()
    if ref is None:
        return None
    frames = [RefFrame(w, ref) for w in wls]
    cores = host_threads()
    # one frame, single thread: sizes the samples
    t1 = time_reference_frames(ref, frames, 1, 1, 1)
    per_thread_fps = 1.0 / t1
    # thread-count sweep: "all the host threads it can use" is whatever count is FASTEST on this box (SMT siblings, a CPU
    # quota of the container or other tenants can make the full logical count slower than a smaller pool)
    curve = {"1": round(per_thread_fps, 3)}
    best_t, best_fps = 1, per_thread_fps
    for t in sorted({8, 16, 32, 64, 96, cores}):
        if t <= 1 or t > cores:
            continue
        n = max(2 * t, min(6 * t, int(0.08 * budget_s * per_thread_fps * t)))
        f = n / time_reference_frames(ref, frames, n, t, t)
        curve[str(t)] = round(f, 3)
        if f > best_fps:
            best_t, best_fps = t, f
    want = max(steps, 6 * best_t)                               # >= 6 frames per thread: the tail wave costs < 15 %
    cap = max(steps, int(0.5 * budget_s * best_fps))            # bounded by the time budget
    n_frames = min(want, cap)
    reps = max(1, -(-n_frames // steps))
    n_frames = reps * steps
    dt = time_reference_frames(ref, frames, n_frames, best_t, warmup)
    out = dict(fps=n_frames / dt, ms=1e3 * dt / n_frames, cores=best_t, host_cpus=cores, tier=REF_TIER_NAME[tier], inner_repeats=reps,
               frames=n_frames, single_thread_fps=per_thread_fps, scaling=curve, cpu_quota=cpu_quota())
    ref.ref_set_threads(best_t)
    return out


def cpu_quota():
    """the container's CPU bandwidth limit (cgroup v2 cpu.max / v1 cfs quota), in CPUs; None = unlimited / unknown"""
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()
        return None if q == "max" else round(int(q) / int(p), 2)
    except Exception:
        pass
    try:
        q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
        p = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
        return None if q <= 0 else round(q / p, 2)
    except Exception:
        return None


# ------------------------------------------------------------------------------------------------------
# clocks sampling (nvidia-smi) during the timed region
# ------------------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock + throttle reasons sampled DURING the timed region: NVML in-process (a sample every ~0.5 ms --
    the timed region is only tens of milliseconds long), nvidia-smi as the fallback."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
    BITS = [0x8, 0x40, 0x20, 0x4]  # nvmlClocksEventReason{HwSlowdown,HwThermalSlowdown,SwThermalSlowdown,SwPowerCap}

    def __init__(self, index, bus_id=None):
        self.samples, self.index, self.stop_flag, self.th = [], index, False, None
        self.nvml = self.handle = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.handle = pynvml.nvmlDeviceGetHandleByPciBusId(bus_id) if bus_id else pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM)
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def _run(self):
        while not self.stop_flag:
            if self.nvml is not None:
                try:
                    mhz = self.nvml.nvmlDeviceGetClockInfo(self.handle, self.nvml.NVML_CLOCK_SM)
                    try:
                        mask = self.nvml.nvmlDeviceGetCurrentClocksEventReasons(self.handle)
                    except Exception:
                        mask = self.nvml.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
                    self.samples.append([str(mhz), str(self.max_mhz)] + ["Active" if mask & b else "Not Active" for b in self.BITS])
                except Exception:
                    pass
                time.sleep(0.0005)
                continue
            try:
                o = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits"],
                                   capture_output=True, text=True, timeout=5).stdout.strip()
                if o:
                    self.samples.append([x.strip() for x in o.split(",")])
            except Exception:
                pass
            time.sleep(0.1)

    def start(self):
        self.th = threading.Thread(target=self._run, daemon=True)
        self.th.start()

    def stop(self):
        self.stop_flag = True
        if self.th:
            self.th.join(timeout=6)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["clock query unavailable"]}
        sm = sorted(int(s[0]) for s in self.samples if s[0].isdigit())
        mx = max(int(s[1]) for s in self.samples if s[1].isdigit())
        reasons = sorted({self.NAMES[i] for s in self.samples for i in range(4) if len(s) > 2 + i and s[2 + i].lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": reasons, "samples": len(self.samples),
                "source": "nvml" if self.nvml is not None else "nvidia-smi"}


# ------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", type=int, default=1, choices=[0, 1, 2, 3, 4], help="BASELINE.json configs[k] (default 1: 1080p 8-bit preset 8)")
    ap.add_argument("--width", type=int, default=0, help="override the configuration's picture size (tests)")
    ap.add_argument("--height", type=int, default=0)
    ap.add_argument("--check", action="store_true", help="compare one frame of B200 output with the reference arm")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--one-stream", action="store_true", help="all frames on one compute stream (no frame-level overlap)")
    ap.add_argument("--e2e-copy-streams", action="store_true",
                    help="end-to-end loop with dedicated copy-in / copy-out streams (default: a frame's copies ride on its own compute stream)")
    ap.add_argument("--streams", type=int, default=4, help="compute streams that consecutive frames alternate between (1, 2, 4 or 8)")
    ap.add_argument("--no-graph", action="store_true", help="launch every kernel eagerly instead of replaying one CUDA graph per step")
    ap.add_argument("--ref-budget", type=float, default=60.0, help="reference arm: upper bound (s) of CPU time for the timed sample")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed to DIR/<name>.npy (B200 arm, rank 0)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the B200 arm")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    warmup = max(args.warmup, 3)

    if args.impl == "reference":
        # the reference's CPU implementation on the host cores; rank 0 alone works, nothing of the product is imported
        if rank != 0:
            return
        W, wls = make_workloads(args, 0, N_FRAME_SETS)
        config = base_config(args, W, wls[0], world, reference=True)
        t = reference_arm(args, wls, args.steps, warmup, budget_s=args.ref_budget)
        if t is None:
            print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/libsvtav1_ref.so is not built"}))
            return
        config["frames_in_flight"] = "one whole frame per host thread, persistent core-pinned pool (%d threads = the fastest count of the sweep on %d host CPUs), %d frame sets" % (t["cores"], t["host_cpus"], N_FRAME_SETS)
        out = {"impl": "reference", "metric": METRIC, "metric_scope": METRIC_SCOPE, "value": round(t["fps"], 3), "unit": "frames/s",
               "n_gpus": args.gpus, "steps": args.steps, "warmup": warmup, "inner_repeats": t["inner_repeats"],
               "ms_per_step": round(t["ms"], 4), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
               "dtype": "u8" if wls[0].bit_depth == 8 else "u16", "data": "synthetic", "config": config,
               "cpu_baseline": {"value": round(t["fps"], 3), "unit": "frames/s", "cores": t["cores"], "kind": "reference",
                                "sample": "%d whole frames in flight over %d pinned threads (%d x %d steps), tier %s" %
                                          (t["frames"], t["cores"], t["inner_repeats"], args.steps, t["tier"]),
                                "scaling": t.get("scaling"), "host_cpus": t["host_cpus"], "cpu_quota": t["cpu_quota"],
                                "single_thread_ms_per_frame": round(1e3 / t["single_thread_fps"], 2)},
               "e2e": {"value": round(t["fps"], 3), "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(out))
        return

    import svt_av1_psy_b200  # noqa: F401  (ImportError = library not built: there is no fallback)
    import torch
    import torch.distributed as dist
    from svt_av1_psy_b200 import dsp, sharding
    from svt_av1_psy_b200.pipeline import FramePipeline
    assert len(FramePipeline.CALLS) == N_CALLS
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        import datetime
        # a mismatched exchange must fail within minutes, not hang the box
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank), timeout=datetime.timedelta(seconds=180))
    dsp.init(local_rank)
    W, wls = make_workloads(args, rank, N_FRAME_SETS)
    wl0 = wls[0]
    config = base_config(args, W, wl0, world, reference=False)
    sets = [FramePipeline(w, torch) for w in wls]
    stream = torch.cuda.Stream()
    n_streams = 1 if args.one_stream else args.streams
    assert n_streams in (1, 2, 4, 8), "--streams must divide the %d frame sets" % N_FRAME_SETS
    streams = [stream] + [torch.cuda.Stream() for _ in range(n_streams - 1)]
    # reconstructed-reference exchange (the path's one real exchange, SURVEY 8e): owner -> consumers, batched per
    # mini-GOP of EXCH_BATCH pictures, on a dedicated communication stream
    comm = torch.cuda.Stream() if world > 1 else None
    exch = sharding.ReconExchange(dist, rank, world, sets[0].final, EXCH_BATCH) if world > 1 else None

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    graphs = [None] * N_FRAME_SETS

    def enqueue_step(i, events=None):
        """one frame of hot-path work on the current stream: replay of the frame set's CUDA graph (the kernel
        launches of a step captured once; same kernels, same work) or, for per-call timing, eager"""
        g = graphs[i % N_FRAME_SETS]
        if g is not None and events is None:
            g.replay()
        else:
            sets[i % N_FRAME_SETS].step(events)

    def capture_graphs():
        for k, fp in enumerate(sets):
            # one eager step on the stream the graph will be captured on: every lazily allocated library
            # workspace (they are per stream) exists before the capture, which must not allocate
            with torch.cuda.stream(streams[k % n_streams]):
                fp.step()
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=streams[k % n_streams]):
                fp.step()
            graphs[k] = g

    class Exchanger:
        """per timed loop: hands every finished picture to the communication stream in mini-GOP batches and keeps
        a frame set from being overwritten before its picture has left"""
        def __init__(self, n):
            self.done = [torch.cuda.Event() for _ in range(n)]
            self.sent = {}     # batch index -> event recorded on the comm stream after the batch's exchange
            self.works = []

        def before_step(self, i, cs):
            j = i - N_FRAME_SETS
            if exch is not None and j >= 0 and (j // EXCH_BATCH) in self.sent:
                cs.wait_event(self.sent[j // EXCH_BATCH])

        def after_step(self, i, cs, n):
            if exch is None:
                return
            self.done[i].record(cs)
            if (i + 1) % EXCH_BATCH == 0 or i == n - 1:
                b0 = (i // EXCH_BATCH) * EXCH_BATCH
                with torch.cuda.stream(comm):
                    for k in range(b0, i + 1):
                        comm.wait_event(self.done[k])
                    self.works += exch.post([sets[k % N_FRAME_SETS].final for k in range(b0, i + 1)])
                    exch.wait(self.works)  # (stream-ordered) the comm stream continues after the group has completed
                    self.works = []
                    ev = torch.cuda.Event()
                    ev.record(comm)
                    self.sent[i // EXCH_BATCH] = ev

        def finish(self, main):
            if exch is not None:
                main.wait_stream(comm)

    def run(n, stage_acc=None):
        ev = [[torch.cuda.Event(enable_timing=True) for _ in range(N_CALLS + 1)] for _ in range(n)] if stage_acc is not None else None
        start, end, tail = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True), torch.cuda.Event()
        ex = Exchanger(n)
        start.record(stream)
        for x in streams[1:]:
            x.wait_event(start)
        if comm is not None:
            comm.wait_event(start)
        for i in range(n):
            st = stream if ev else streams[i % n_streams]  # the per-call profile runs strictly serially
            with torch.cuda.stream(st):
                ex.before_step(i, st)
                enqueue_step(i, ev[i] if ev else None)
                ex.after_step(i, st, n)
        for x in streams[1:]:
            tail.record(x)
            stream.wait_event(tail)
        ex.finish(stream)
        end.record(stream)
        torch.cuda.synchronize()
        if stage_acc is not None:  # per call: n x the MEDIAN over the steps (one slow first launch must not pose as the dominant call)
            for k in range(N_CALLS):
                v = sorted(ev[i][k].elapsed_time(ev[i][k + 1]) for i in range(n))
                stage_acc[k] += n * v[len(v) // 2]
        return start.elapsed_time(end)

    s_in, s_out = torch.cuda.Stream(), torch.cuda.Stream()

    host_enqueue = [0.0, 0]  # seconds the host spent enqueueing e2e frames, frames
    D2H_LAG = 5  # the variable-size part of a frame's results is requested this many frames later (its size has arrived by then; < N_FRAME_SETS)
    d2h_level_bytes = [0, 0]  # bytes, frames

    def run_e2e(n):
        """host buffers -> device -> host, every step: copy-in, graph replay and copy-out of a frame are enqueued back to back on
        the frame's compute stream (consecutive frames use different streams, so the three phases of different frames overlap);
        a frame set is re-used only after its previous results have been read back (same stream, later).  --e2e-copy-streams
        uses dedicated copy streams ordered with events instead.  Results travel in two parts: the fixed-size outputs
        (with the level offsets), then -- D2H_LAG frames later, when the host knows sum(eob) -- exactly that many levels."""
        ev_in = [torch.cuda.Event() for _ in range(n)]
        ev_done = [torch.cuda.Event() for _ in range(n)]
        ev_small = [torch.cuda.Event() for _ in range(n)]
        ev_out = [torch.cuda.Event() for _ in range(n)]
        ex = Exchanger(n)
        start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

        h_in, h_out = s_in.cuda_stream, s_out.cuda_stream

        def finish_frame(k):
            ev_small[k].synchronize()  # host wait, but on work enqueued D2H_LAG frames ago: the pipeline stays full
            d2h_level_bytes[0] += sets[k % N_FRAME_SETS].read_levels(h_out)
            d2h_level_bytes[1] += 1
            ev_out[k].record(s_out)

        t_host = time.perf_counter()
        start.record(stream)
        if not args.e2e_copy_streams:
            # default: a frame's copy-in, its graph replay and its copy-out are enqueued on the frame's own compute stream (frames
            # alternate between the compute streams, so the copies of one frame still overlap the kernels of the others); the host
            # issues 3 library calls + 1 event per frame
            def finish_frame(k):  # noqa: F811
                ev_small[k].synchronize()  # host wait, but on work enqueued D2H_LAG frames ago: the pipeline stays full
                cs = streams[k % n_streams]
                d2h_level_bytes[0] += sets[k % N_FRAME_SETS].read_levels(cs.cuda_stream)
                d2h_level_bytes[1] += 1
            for x in streams[1:]:
                x.wait_event(start)
            if comm is not None:
                comm.wait_event(start)
            for i in range(n):
                fp = sets[i % N_FRAME_SETS]
                cs = streams[i % n_streams]
                with torch.cuda.stream(cs):
                    ex.before_step(i, cs)
                    fp.load_inputs(cs.cuda_stream)
                    enqueue_step(i)
                    ex.after_step(i, cs, n)
                    fp.read_outputs(cs.cuda_stream)
                    ev_small[i].record(cs)
                if i >= D2H_LAG:
                    finish_frame(i - D2H_LAG)
            for k in range(max(0, n - D2H_LAG), n):
                finish_frame(k)
            tail = torch.cuda.Event()
            for x in streams[1:]:
                tail.record(x)
                stream.wait_event(tail)
            ex.finish(stream)
            end.record(stream)
            host_enqueue[0] += time.perf_counter() - t_host
            host_enqueue[1] += n
            torch.cuda.synchronize()
            return start.elapsed_time(end)
        # --e2e-copy-streams: dedicated copy-in / copy-out streams, ordered with events (more host work per frame)
        s_in.wait_event(start)
        if comm is not None:
            comm.wait_event(start)
        for i in range(n):
            fp = sets[i % N_FRAME_SETS]
            if i >= N_FRAME_SETS:
                s_in.wait_event(ev_out[i - N_FRAME_SETS])
                ex.before_step(i, s_in)
            fp.load_inputs(h_in)
            ev_in[i].record(s_in)
            cs = streams[i % n_streams]
            cs.wait_event(ev_in[i])
            with torch.cuda.stream(cs):
                enqueue_step(i)
            ev_done[i].record(cs)
            ex.after_step(i, cs, n)
            s_out.wait_event(ev_done[i])
            fp.read_outputs(h_out)
            ev_small[i].record(s_out)
            if i >= D2H_LAG:
                finish_frame(i - D2H_LAG)
        for k in range(max(0, n - D2H_LAG), n):
            finish_frame(k)
        stream.wait_event(ev_out[n - 1])
        ex.finish(stream)
        end.record(stream)
        host_enqueue[0] += time.perf_counter() - t_host
        host_enqueue[1] += n
        torch.cuda.synchronize()
        return start.elapsed_time(end)

    if args.check and rank == 0:
        check_against_reference(sets[0], torch)

    # ---- resident-input timing ---------------------------------------------------------------------------
    run(warmup)
    barrier()
    # per-call profile: eager launches with an event around every T2 call (not part of the timed value)
    l0 = dsp.launch_count()
    call_ms = [0.0] * N_CALLS
    prof_steps = min(args.steps, 40)
    ms_eager = run(prof_steps, call_ms)
    launches_per_step = (dsp.launch_count() - l0) / prof_steps
    if not args.no_graph:
        capture_graphs()
        run(warmup)
    barrier()
    bus_id = None
    try:  # NVML enumerates physical devices: address this rank's GPU by PCI id, not by (visible) index
        pr = torch.cuda.get_device_properties(local_rank)
        bus_id = "%08X:%02X:%02X.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
    except Exception:
        bus_id = None
    sampler = ClockSampler(local_rank, bus_id)
    sampler.start()
    ms = run(args.steps)
    barrier()
    # ---- end-to-end timing -----------------------------------------------------------------------------------
    run_e2e(warmup)
    barrier()
    ms_e2e = run_e2e(args.steps)
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(sets[(args.steps - 1) % N_FRAME_SETS], args.dump_outputs)
    t = torch.tensor([ms, ms_e2e], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, ms_e2e = float(t[0]), float(t[1])
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    fps = world * args.steps / (ms / 1e3)
    fps_e2e = world * args.steps / (ms_e2e / 1e3)
    alg = wl0.algorithmic_bytes()
    call_ms = [x / prof_steps for x in call_ms]
    calls = FramePipeline.CALLS
    names = list(FramePipeline.STAGES)
    stage_ms = [sum(call_ms[i] for i, c in enumerate(calls) if c[1] == st) for st in names]
    dom = int(np.argmax(call_ms))
    dom_name, _, dom_kernels = calls[dom]
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    src = "MEASURED_PEAKS.json" if peaks else "built-in defaults"
    ncu_bytes, ncu_src = ncu_dram_bytes(args.config, dom_name) if not args.width else (None, None)
    if dom_name == "wiener_stats":  # the one dense contraction of the path: exact f16 MMA on the tensor cores
        flops = 2.0 * wl0.wiener_stats_macs()
        peak = float(peaks.get("bf16_tflops", peaks.get("dense_bf16_tflops", 2250.0)))
        ach = flops / (call_ms[dom] / 1e3) / 1e12
        roofline = {"bound": "tensor", "achieved": round(ach, 3), "peak": peak, "unit": "TFLOP/s", "frac": round(ach / peak, 5),
                    "algorithmic_flops_per_call": flops}
    else:
        peak = float(peaks.get("hbm_gbs", 6650.0))
        ach = alg[dom_name] / (call_ms[dom] / 1e3) / 1e9
        roofline = {"bound": "hbm", "achieved": round(ach, 2), "peak": peak, "unit": "GB/s", "frac": round(ach / peak, 5),
                    "algorithmic_bytes_per_call": alg[dom_name],
                    "note": "integer kernel working out of shared-memory tiles: instruction/latency bound, not HBM bound (SURVEY 8d)"}
        if dom_name == "txfm_trio":  # SURVEY 8(d)'s figure counts the unfused chain's intermediates; what the fused call must move is less
            fm = alg["txfm_trio_fused_min"]
            roofline["fused_min_bytes_per_call"] = fm
            roofline["frac_fused_min"] = round(fm / (call_ms[dom] / 1e3) / 1e9 / peak, 5)
    roofline.update({"call": dom_name, "kernel": dom_kernels, "ms_per_call": round(call_ms[dom], 4), "peak_source": src,
                     "traffic": ncu_bytes, "traffic_source": ("%s (ncu launch list of tools/profile_step.py, DRAM read + write of the call's kernels)" % ncu_src) if ncu_bytes is not None else None})
    out = {"metric": METRIC, "value": round(fps, 2), "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": warmup,
           "timed_region_ms": round(ms, 3),
           "ms_per_step": round(ms / args.steps, 4), "metric_scope": METRIC_SCOPE, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
           "dtype": "u8" if wl0.bit_depth == 8 else "u16",
           "data": "synthetic", "config": config, "clocks": clocks,
           "e2e": {"value": round(fps_e2e, 2), "unit": "frames/s", "h2d_bytes_per_step": int(sets[0].h2d_bytes),
                   "d2h_bytes_per_step": int(sets[0].d2h_fixed_bytes + d2h_level_bytes[0] / max(1, d2h_level_bytes[1])),
                   "d2h_note": "fixed-size results + sum(eob) scan-order levels (%d-byte), averaged over the timed frames" % sets[0].level_bytes,
                   "ms_per_step": round(ms_e2e / args.steps, 4),
                   "host_enqueue_ms_per_step": round(1e3 * host_enqueue[0] / max(1, host_enqueue[1]), 4)},
           "gpu_launches": int(round(launches_per_step * args.steps)), "gpu_launches_per_step": round(launches_per_step, 1),
           # serial sum of the per-call medians (the eager loop's wall time also holds one-off first-launch costs)
           "eager_ms_per_step": round(sum(call_ms), 4), "eager_loop_ms_per_step": round(ms_eager / prof_steps, 4), "roofline": roofline,
           "stages_ms": {n: round(v, 4) for n, v in zip(names, stage_ms)},
           "calls_ms": {c[0]: round(v, 4) for c, v in zip(calls, call_ms)},
           "calls_algorithmic_gbs": {c[0]: round(alg[c[0]] / (v / 1e3) / 1e9, 2) for c, v in zip(calls, call_ms) if v > 0}}
    if world > 1:
        out["exchange"] = {"pattern": "owner -> %d consumers (point-to-point), batched per %d pictures, dedicated comm stream" % (len(exch.consumers), EXCH_BATCH),
                           "bytes_sent_per_step_per_rank": int(exch.bytes_sent_per_frame)}
    if world == 1 and not args.no_cpu_baseline:
        t = reference_arm(args, wls, args.steps, 3, budget_s=min(args.ref_budget, 20.0))
        if t is not None:
            out["cpu_baseline"] = {"value": round(t["fps"], 3), "unit": "frames/s", "cores": t["cores"], "kind": "reference",
                                   "sample": "%d whole frames of the same workload in flight over %d pinned host threads (fastest count on %d CPUs), tier %s" %
                                             (t["frames"], t["cores"], t["host_cpus"], t["tier"]), "scaling": t["scaling"]}
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


DUMP_BYTES = 64 << 20


def dump_outputs(fp, out_dir):
    """What the caller of the timed path receives for the frame of `fp`'s last step: the read-back results (ME results, eobs, level
    offsets, CDEF costs, Wiener statistics), the sum(eob) packed levels and the restored picture.  Written as <name>.npy, float32
    for values of up to 16 bits and float64 otherwise (exact either way); an array larger than its share of DUMP_BYTES is
    replaced by a fixed seeded sample of its elements (sorted flat indices, the same in every run of the same arguments)."""
    import torch
    torch.cuda.synchronize()
    arrays = {k: v.numpy() for k, v in fp.h_out.items()}
    arrays["levels"] = fp.h_levels.numpy()[:int(arrays["level_offsets"][fp.n_tx])]
    arrays["final"] = fp.final.cpu().numpy()
    os.makedirs(out_dir, exist_ok=True)
    share = DUMP_BYTES // len(arrays)
    for name, a in sorted(arrays.items()):
        a = a.astype(np.float32 if a.dtype.itemsize <= 2 else np.float64).reshape(-1)
        n = share // a.itemsize
        if a.size > n:
            a = a[np.sort(np.random.default_rng(20260923).choice(a.size, n, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def base_config(args, W, wl, world, reference):
    cfg = {"workload": W.CONFIG_NAMES[args.config], "width": wl.width, "height": wl.height, "bit_depth": wl.bit_depth, "preset": wl.preset,
           "frame_sets": N_FRAME_SETS,
           "l2": "steps rotate over %d distinct frame sets (>= 65 MB each, > the 126 MB L2 in total)" % N_FRAME_SETS,
           "parallelism": "frame-parallel x%d (no data-path collective; reconstructed reference pictures go owner -> consumers)" % world}
    if not reference:
        cfg.update({"overlap": "ME (source pictures only) on a side stream, concurrent with the transform->CDEF->restoration chain of the same step",
                    "streams": "1 compute stream" if args.one_stream else "%d compute streams: consecutive (independent) frames alternate between them" % args.streams,
                    "launch": "eager" if args.no_graph else "one CUDA graph replay per step (the step's kernel launches captured once per frame set)"})
    return cfg


def reference_frame(wl):
    """the reference arm's outputs for one frame of `wl` (default seed): name -> array where oracle/_ref is built, else
    name -> the SHA-256 of those bytes as committed in tests/golden/frame_<W>x<H>[_b<bd>_m<preset>].json (tools/make_golden.py)"""
    ref, _ = load_reference()
    if ref is None:
        name = "frame_%dx%d%s.json" % (wl.width, wl.height, "" if (wl.bit_depth, wl.preset) == (8, 8) else "_b%d_m%d" % (wl.bit_depth, wl.preset))
        path = os.path.join(ROOT, "tests", "golden", name)
        assert os.path.isfile(path), "no reference digests for this frame (%s) and oracle/_ref is not built" % name
        return json.load(open(path))["sha256"]
    from oracle.frame_ref import RefFrame
    from svt_av1_psy_b200.layout import ME_OUTPUT_NAMES
    ref.ref_set_tier(0)
    fr = RefFrame(wl, ref)
    fr.step()
    ref.ref_set_tier(1)
    out = {k: fr.me[f] for k, f in ME_OUTPUT_NAMES.items()}
    out.update({"residual": fr.residual, "coeff": fr.coeff, "qcoeff": fr.q, "dqcoeff": fr.dq, "eob": fr.eobs, "recon": fr.recon,
                "cdef_mse": fr.mse, "cdef_dir": fr.dirs, "cdef_out": fr.cdef_out, "wiener_M": fr.M, "wiener_H": fr.Hm, "final": fr.final})
    return out


def check_against_reference(fp, torch):
    """one frame through both arms, every output compared bit for bit (through its digest where oracle/_ref is not built)"""
    import hashlib
    want = reference_frame(fp.wl)
    fp.load_inputs()
    fp.step()
    torch.cuda.synchronize()
    from svt_av1_psy_b200.layout import ME_OUTPUT_NAMES
    cmp = [(k, fp.me[f]) for k, f in ME_OUTPUT_NAMES.items()] + [
           ("qcoeff", fp.qcoeff), ("dqcoeff", fp.dqcoeff), ("eob", fp.eobs), ("recon", fp.recon), ("cdef_mse", fp.cdef_mse),
           ("cdef_dir", fp.cdef_dir), ("cdef_out", fp.cdef_out), ("wiener_M", fp.M), ("wiener_H", fp.Hm), ("final", fp.final)]
    bad = []

    def compare(items, tag=""):
        for name, a in items:
            a = np.ascontiguousarray(a.cpu().numpy()).view(np.uint8).reshape(-1)
            b = want[name]
            same = hashlib.sha256(a).hexdigest() == b if isinstance(b, str) else np.array_equal(a, np.ascontiguousarray(b).view(np.uint8).reshape(-1))
            if not same:
                bad.append(name + tag)

    compare(cmp)
    # the packed levels: block i's first eob levels in scan order at offsets[i] == what the entropy coder reads from the reference's
    # buffers (the eobs and quantized coefficients, compared with the reference's above)
    offs = fp.level_offsets.cpu().numpy().view(np.uint32)
    lv = fp.levels.cpu().numpy()
    eobs = fp.eobs.cpu().numpy().reshape(-1).astype(np.int64)
    q = fp.qcoeff.cpu().numpy().reshape(-1)
    want_offs = np.concatenate([[0], np.cumsum(eobs)])
    if not np.array_equal(offs[:len(want_offs)], want_offs) or offs[len(want_offs)] != 0:
        bad.append("level_offsets")
    else:
        qi, scan = fp.wl.quant_items, fp.wl.scan_table
        for i in range(0, len(qi), max(1, len(qi) // 4000)):  # every block of a small picture, a dense sample of a large one
            e = int(eobs[i])
            w = q[int(qi["q_off"][i]) + scan[int(qi["scan_off"][i]):int(qi["scan_off"][i]) + e].astype(np.int64)]
            if not np.array_equal(lv[want_offs[i]:want_offs[i] + e].astype(np.int64), w.astype(np.int64)):
                bad.append("levels[block %d]" % i)
                break
    # the frame step uses the fused transform call; the same chain as three separate calls (which also
    # materialises the forward coefficients) must give the same answers
    s = torch.cuda.current_stream().cuda_stream
    for t in (fp.qcoeff, fp.dqcoeff, fp.eobs, fp.recon, fp.residual):
        t.zero_()
    fp.call_residual(s)
    fp.call_fwd_txfm(s)
    fp.call_quant(s)
    fp.call_inv_txfm(s)
    torch.cuda.synchronize()
    split = [("residual", fp.residual), ("coeff", fp.coeff), ("qcoeff", fp.qcoeff), ("dqcoeff", fp.dqcoeff), ("eob", fp.eobs), ("recon", fp.recon)]
    compare(split, "/3-call")
    n = len(cmp) + len(split)
    if bad:
        raise SystemExit("PARITY FAILURE vs reference: " + ", ".join(bad))
    print("parity vs reference C tier%s: all %d outputs bit-exact" % (" (committed digests)" if isinstance(want["final"], str) else "", n), file=sys.stderr)
    return n


if __name__ == "__main__":
    main()
