"""Aided search against the full search on one GPU (acq_search_aided / acq_search_aided_device).

  cfg1 : one capture, 32 PRNs through the host path -- end-to-end call latency of acq_search (41 bins) and of
         acq_search_aided with W = 3, 5, 9; median over >= 2000 calls each after warm-up, the four calls interleaved.
  cfg5 : the 1024-capture receiver farm (bench.farm_captures_numpy) on the device path, full search against W = 5,
         centres = true Doppler of the injected signals + a seeded offset in +-2 (a seeded random index for satellites
         without a signal).  Device step time by CUDA events, full and aided steps interleaved on the same captures;
         tiles/s and cells examined per second.

Records the GPU's name, power limit and maximum SM clock (nvidia-smi query) in the same run and writes
<out>/aided_bench_<tag>.json.  Usage: python tools/aided_bench.py --tag b200 [--out profiles]
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


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown (%s)" % q.stderr.strip()


def cfg1(F, S, synth, scenarios, calls, warmup):
    table = S.navstar()
    cap = np.ascontiguousarray(synth.make_capture(10_005, 1, table, scenarios.signals("cfg1", 1)))
    out = np.zeros(32, F.RECORD_DTYPE)
    rng = np.random.default_rng(1)
    centers = rng.integers(-20, 21, 32).astype(np.int32)
    res = {}
    with F.AcqEngine(table) as eng:
        L, h = eng._L, eng._h
        cp, op, ccp = cap.ctypes.data, out.ctypes.data, centers.ctypes.data
        calls_of = {"full_41": lambda: L.acq_search(h, cp, 1, None, 0, op)}
        for hw in (1, 2, 4):
            calls_of["aided_W%d" % (2 * hw + 1)] = (lambda hw=hw: L.acq_search_aided(h, cp, 1, None, 0, ccp, hw, op, None))
        times = {k: [] for k in calls_of}
        for k, fn in calls_of.items():
            for _ in range(warmup):
                assert fn() == 0, L.acq_last_error()
        rounds = 10
        for _ in range(rounds):   # the four calls interleaved in blocks, so clock drift touches all alike
            for k, fn in calls_of.items():
                t = times[k]
                for _ in range(calls // rounds):
                    t0 = time.perf_counter_ns()
                    rc = fn()
                    t.append(time.perf_counter_ns() - t0)
                    assert rc == 0
        for k, t in times.items():
            t = np.array(t) / 1e3
            res[k] = {"calls": len(t), "median_us": float(np.median(t)), "p10_us": float(np.percentile(t, 10)),
                      "p90_us": float(np.percentile(t, 90))}
    return res


def farm_centers(F, bench, n_cap, n_sel):
    """Doppler centres of the farm's aided search: the true Doppler of each injected signal + a seeded offset in +-2, a
    seeded random index for satellites without a signal."""
    rng = np.random.default_rng(5)
    centers = rng.integers(-20, 21, (n_cap, n_sel)).astype(np.int32)
    for c in range(n_cap):
        for sat, _, f, _, _ in bench.farm_signals(c):
            centers[c, sat] = int(np.round(f / F.BIN_HZ)) + int(rng.integers(-2, 3))
    return centers


def cfg5(F, S, torch, bench, steps):
    table = S.navstar()
    n_cap, n_sel, hw = 1024, 32, 2
    caps = bench.farm_captures_numpy(range(n_cap))
    centers = farm_centers(F, bench, n_cap, n_sel)
    res = {}
    with F.AcqEngine(table) as eng:
        d_in = torch.from_numpy(caps.reshape(-1)).cuda()
        d_c = torch.from_numpy(centers.reshape(-1)).cuda()
        d_full = torch.zeros(n_cap * n_sel * 24, dtype=torch.uint8, device="cuda")
        d_aid = torch.zeros_like(d_full)
        # a non-default stream: its handle is non-NULL, so the engine launches on exactly this stream and the events
        # bracket its kernels (NULL would select the engine's own stream)
        st = torch.cuda.Stream()
        torch.cuda.synchronize()
        runs = {"full_41": lambda: eng.search_device(d_in.data_ptr(), d_full.data_ptr(), n_cap, stream_ptr=st.cuda_stream),
                "aided_W5": lambda: eng.search_aided_device(d_in.data_ptr(), d_c.data_ptr(), hw, d_aid.data_ptr(), n_cap,
                                                            stream_ptr=st.cuda_stream)}
        ms = {k: [] for k in runs}
        for k, fn in runs.items():   # warm-up
            for _ in range(3):
                fn()
        torch.cuda.synchronize()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        for _ in range(steps):
            for k, fn in runs.items():   # interleaved on the same captures
                ev[0].record(st)
                fn()
                ev[1].record(st)
                ev[1].synchronize()
                ms[k].append(ev[0].elapsed_time(ev[1]))
        # per-kernel split (engine profiling: event records between the kernels, so no programmatic dependent launch)
        eng.set_profiling(True)
        kern = {k: [] for k in runs}
        for _ in range(5):
            for k, fn in runs.items():
                fn()
                kern[k].append(eng.kernel_ms())
        eng.set_profiling(False)
        full = d_full.cpu().numpy().view(F.RECORD_DTYPE).reshape(n_cap, n_sel)
        aid = d_aid.cpu().numpy().view(F.RECORD_DTYPE).reshape(n_cap, n_sel)
    for k, W in (("full_41", 41), ("aided_W5", 5)):
        m = statistics.median(ms[k])
        tiles = n_cap * n_sel * W
        res[k] = {"steps": len(ms[k]), "median_ms": m, "min_ms": min(ms[k]), "max_ms": max(ms[k]), "tiles": tiles,
                  "tiles_per_s": tiles / (m * 1e-3), "cells_per_s": tiles * F.LAGS_L1 / (m * 1e-3)}
        km = {n: statistics.median(x[n] for x in kern[k]) for n in kern[k][0]}
        res[k]["kernel_ms_profiled"] = km
        res[k]["search_kernel_tiles_per_s"] = tiles / (km["search"] * 1e-3)
    # injected satellites the full search detects: where its pick lies inside the row's window the aided record must be
    # the same bytes; outside (the true bin's neighbour won the full search, the window is off by the other side) not
    det_full = det_in = det_same = 0
    for c in range(n_cap):
        for sat, _, _, _, _ in bench.farm_signals(c):
            if full[c, sat]["snr"] >= 16:
                det_full += 1
                lo = min(max(int(centers[c, sat]) - hw, -20), 20 - 2 * hw)
                if lo <= full[c, sat]["dop"] <= lo + 2 * hw:
                    det_in += 1
                    det_same += int(aid[c, sat].tobytes() == full[c, sat].tobytes())
    res["detections"] = {"detected_by_full": det_full, "full_pick_inside_window": det_in, "aided_record_identical": det_same}
    res["l2"] = "not flushed between steps: full and aided steps alternate on the same 1024 captures"
    res["speedup_step"] = res["full_41"]["median_ms"] / res["aided_W5"]["median_ms"]
    res["tile_rate_ratio"] = res["aided_W5"]["tiles_per_s"] / res["full_41"]["tiles_per_s"]
    res["search_kernel_tile_rate_ratio"] = res["aided_W5"]["search_kernel_tiles_per_s"] / res["full_41"]["search_kernel_tiles_per_s"]
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--tag", default="b200")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"))
    ap.add_argument("--calls", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=300)
    ap.add_argument("--steps", type=int, default=30)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("aided_bench: no CUDA device (nothing is measured without one)")
    import bench
    import flydog_sdr_gps_b200 as F
    from flydog_sdr_gps_b200 import scenarios, synth
    from flydog_sdr_gps_b200 import sats as S
    result = {"gpu": gpu_info(), "torch_gpu": torch.cuda.get_device_name(0),
              "cfg1": cfg1(F, S, synth, scenarios, args.calls, args.warmup),
              "cfg5": cfg5(F, S, torch, bench, args.steps)}
    result["gpu_after"] = gpu_info()
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "aided_bench_%s.json" % args.tag)
    with open(path, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result))


if __name__ == "__main__":
    main()
