#!/usr/bin/env python3
"""Times the Wiener statistics call (svt_b200_compute_stats_batch_dev) alone on the statistics items of bench.py
configurations: CUDA events around many back-to-back launches that rotate over frame sets whose planes together
exceed twice the L2, so no launch finds its pixels there.

  python tools/bench_stats.py [--configs 1 3] [--iters 400] [--warmup 40]

Prints the card name and power limit first, then per configuration: ms per frame, useful MAC/s (the reference's
win^2 (win^2 + 1) / 2 + win^2 multiply-accumulates per pixel) and, for 8-bit pictures, the MAC/s the tensor-core
kernel issues, both next to the data-sheet dense INT8 rate of one B200.  stats_mma_kernel (wiener.cu) issues one
M = N = 128, K = 32 MMA per block of up to T output rows and 32 columns of a tile, T = 10 / 12 / 14 at WIN 7 / 5 / 3,
in tiles of 30 / 36 / 28 rows: a tile of r rows takes ceil(r / T) blocks."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

INT8_DENSE_MACS = 4.5e15 / 2  # HGX B200 data sheet, one GPU, dense INT8 (ops = 2 MAC)


def card():
    import torch
    q = ["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"]
    try:
        smi = subprocess.run(q, capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.TimeoutExpired) as e:
        smi = "nvidia-smi unavailable (%s)" % e
    return {"device": torch.cuda.get_device_name(0), "name,power.limit,clocks.max.sm": smi}


def block_rows(win):
    """output rows per MMA (stats_block_rows in wiener.cu) and rows per tile (stats_tile_rows)"""
    t = (127 - 9 * (win - 1)) // 8 + 1
    return t, t * (36 // t)


def issued_macs(items):
    tot = 0
    for it in items:
        win, w, h = int(it["wiener_win"]), int(it["h_end"]) - int(it["h_start"]), int(it["v_end"]) - int(it["v_start"])
        t, th = block_rows(win)
        blocks = sum(-(-min(th, h - y) // t) for y in range(0, h, th))  # per column of tiles
        tot += blocks * ((w + 31) // 32) * 128 * 128 * 32
    return tot


def run(k, iters, warmup):
    import numpy as np
    import torch
    from svt_av1_psy_b200.dsp import lib
    from svt_av1_psy_b200.workload import CONFIGS, FrameWorkload

    w, h, bd, preset = CONFIGS[k]
    wl = FrameWorkload(w, h, bit_depth=bd, preset=preset)
    n_dgd, n_src = wl.padded_offsets()[1], wl.flat_offsets()[1]
    set_bytes = (n_dgd + n_src) * wl.pixel_bytes
    l2 = torch.cuda.get_device_properties(0).L2_cache_size
    n_sets = max(8, -(-2 * l2 // set_bytes))
    dt = torch.uint8 if bd == 8 else torch.int16
    gen = torch.Generator(device="cuda").manual_seed(k)
    sets = [tuple(torch.randint(0, 1 << bd, (n,), dtype=dt, device="cuda", generator=gen) for n in (n_dgd, n_src)) for _ in range(n_sets)]
    items = torch.from_numpy(wl.stats_items.view(np.uint8).copy()).cuda()
    n = len(wl.stats_items)
    M = torch.empty((n, 49), dtype=torch.int64, device="cuda")
    H = torch.empty((n, 2401), dtype=torch.int64, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream

    def call(i):
        dgd, src = sets[i % n_sets]
        rc = lib.svt_b200_compute_stats_batch_dev(dgd.data_ptr(), src.data_ptr(), items.data_ptr(), n, bd, M.data_ptr(), H.data_ptr(), stream)
        if rc != 0:
            raise RuntimeError("svt_b200_compute_stats_batch_dev returned %d" % rc)

    for i in range(warmup):
        call(i)
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for i in range(iters):
        call(i)
    t1.record()
    torch.cuda.synchronize()
    ms = t0.elapsed_time(t1) / iters
    useful = wl.wiener_stats_macs()
    out = {"config": k, "picture": "%dx%d %d-bit" % (w, h, bd), "items": n, "frame_sets": n_sets, "set_mb": round(set_bytes / 1e6, 1),
           "iters": iters, "ms_per_frame": round(ms, 4), "useful_gmac": round(useful / 1e9, 3),
           "useful_tmac_s": round(useful / ms / 1e9, 2), "int8_dense_tmac_s": INT8_DENSE_MACS / 1e12}
    if bd == 8:
        issued = issued_macs(wl.stats_items)
        out.update({"issued_gmac": round(issued / 1e9, 3), "issued_tmac_s": round(issued / ms / 1e9, 2),
                    "issued_share_of_int8_dense": round(issued / ms * 1e3 / INT8_DENSE_MACS, 4)})
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", type=int, nargs="+", default=[1, 3])
    ap.add_argument("--iters", type=int, default=400)
    ap.add_argument("--warmup", type=int, default=40)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_stats.py needs a CUDA device")
    import svt_av1_psy_b200 as pkg
    pkg.init(0)
    print(json.dumps(card()))
    for k in args.configs:
        print(json.dumps(run(k, args.iters, args.warmup)))


if __name__ == "__main__":
    main()
