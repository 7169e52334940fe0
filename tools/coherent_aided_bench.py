"""Aided coherent search (acq_search_coherent_aided) against the full coherent search on one GPU.

  throughput   the cfg2 shape (coherent_bench.CFG2: K = 20, half-bins, +-80) over 128 captures x 32 PRNs through the
               device forms, at M = 4 and 5: the full coherent search against windows of +-1, +-2 and +-4 engine
               half-bins (half_width = M, 2M, 4M coherent steps).  Search-kernel time (the engine's CUDA events around
               the search launch, acq_set_profiling) and the whole search (CUDA events on a non-default stream);
               block-IFFTs per second (captures x 32 x cells x K over the search-kernel time); the time per block-IFFT
               relative to the full coherent search; and the fixed part no window shrinks: front end with k_coh_variants
               and the forward FFT of F variants per block.  The capture spectra (2560 blocks x F variants x 128 KiB)
               exceed the 126 MB L2, so L2 is not flushed between calls.
  latency      one capture, 32 PRNs, a K = 4 engine (full bins, +-20), M = 4 through the host forms: per-call time of
               acq_search_coherent_aided with half_width 4 and 8 against acq_search_coherent and acq_search (host clock
               around the synchronous calls, medians after warm-up, calls interleaved).
  sensitivity  coherent_bench's sensitivity set at 27 / 29 / 31 dB-Hz, M = 1, 4 and 5, full coherent search against the
               aided one with centres at the true Doppler's coherent index plus a seeded offset of at most M steps and
               half_width = 2M; and the snr quantiles (50 / 99 / 99.9 %) of noise-only captures per (M, W), from which a
               threshold for a windowed search can be chosen.

Records the GPU's name, power limit and maximum SM clock (nvidia-smi query) in the same run and writes
<out>/coherent_aided_bench_<tag>.json.  Usage: python tools/coherent_aided_bench.py --tag b200 [--out profiles] [--steps 5]
"""
import argparse
import json
import os
import statistics
import sys
import time

import numpy as np

TOOLS = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(TOOLS)
sys.path.insert(0, ROOT)
sys.path.insert(0, TOOLS)

from aided_bench import gpu_info  # noqa: E402
from coherent_bench import CFG2, found, sensitivity_set  # noqa: E402


def truth_centers(F, eng, m_coh, f_hz, seed):
    """The true Doppler's index on the coherent grid plus a seeded offset in [-M, M] (one engine half-bin)."""
    Fv = m_coh * (1 + eng.params.half_bin)
    h = np.round(np.asarray(f_hz) * Fv / F.BIN_HZ).astype(np.int64)
    return (h + np.random.default_rng(seed).integers(-m_coh, m_coh + 1, h.size)).astype(np.int32)


def throughput(F, S, synth, torch, steps):
    table = S.navstar()
    n_cap, n_sel = 128, 32
    caps, _, _ = sensitivity_set(F, S, synth, torch, 5, n_cap, 30.0)
    res = {}
    with F.AcqEngine(table, F.default_params(**CFG2)) as eng:
        K = eng.k_noncoh
        d_in = torch.from_numpy(caps.reshape(-1)).cuda()
        d_rec = torch.zeros(n_cap * n_sel * 24, dtype=torch.uint8, device="cuda")
        st = torch.cuda.Stream()
        sp = st.cuda_stream
        rng = np.random.default_rng(3)
        calls = {}
        centers = {}
        for m in (4, 5):
            clo, chi = m * eng.params.dop_lo, m * eng.params.dop_hi
            centers[m] = torch.from_numpy(rng.integers(clo, chi + 1, n_cap * n_sel).astype(np.int32)).cuda()
            calls["coherent_m%d" % m] = ((lambda m=m: eng.search_coherent_device(d_in.data_ptr(), m, d_rec.data_ptr(), n_cap,
                                                                                  stream_ptr=sp)),
                                         eng.coherent_dops(m), m, None)
            for k in (1, 2, 4):
                hw = k * m
                calls["aided_m%d_hw%d" % (m, hw)] = (
                    (lambda m=m, hw=hw: eng.search_coherent_aided_device(d_in.data_ptr(), m, centers[m].data_ptr(), hw,
                                                                         d_rec.data_ptr(), n_cap, stream_ptr=sp)),
                    2 * hw + 1, m, hw)
        torch.cuda.synchronize()
        kern = {k: [] for k in calls}
        fixed = {k: [] for k in calls}
        whole = {k: [] for k in calls}
        for k, (fn, _, _, _) in calls.items():
            fn()
        torch.cuda.synchronize()
        for _ in range(steps):
            for k, (fn, _, _, _) in calls.items():   # interleaved; kernel times from the engine's events (profiling on)
                eng.set_profiling(True)
                fn()
                km = eng.kernel_ms()
                kern[k].append(km["search"])
                fixed[k].append(km["front_end"] + km["fwd_fft"])
                eng.set_profiling(False)
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(st)
                fn()
                b.record(st)
                b.synchronize()
                whole[k].append(a.elapsed_time(b))
        for k, (_, n_dop, m, hw) in calls.items():
            ms = statistics.median(kern[k])
            n_ifft = n_cap * n_sel * n_dop * K
            res[k] = {"m_coh": m, "half_width": hw, "cells_per_row": n_dop, "search_kernel_ms": ms,
                      "search_kernel_ms_min": min(kern[k]), "fixed_front_end_variants_fwd_fft_ms": statistics.median(fixed[k]),
                      "whole_search_ms": statistics.median(whole[k]), "block_iffts": n_ifft,
                      "block_iffts_per_s": n_ifft / (ms * 1e-3)}
        for k, (_, n_dop, m, _) in calls.items():
            base = res["coherent_m%d" % m]
            res[k]["time_per_block_ifft_vs_full_coherent"] = (res[k]["search_kernel_ms"] / res[k]["block_iffts"]) / (
                base["search_kernel_ms"] / base["block_iffts"])
            res[k]["search_kernel_ms_vs_full_coherent"] = res[k]["search_kernel_ms"] / base["search_kernel_ms"]
            res[k]["whole_search_ms_vs_full_coherent"] = res[k]["whole_search_ms"] / base["whole_search_ms"]
    return res


def latency(F, S, synth, steps):
    table = S.navstar()
    cap = np.ascontiguousarray(synth.make_capture(4711, 4, table, [(3, 4000, 3.4 * F.BIN_HZ, 44, 0.5)]))
    M = 4
    res = {}
    with F.AcqEngine(table, F.default_params(k_noncoh=4)) as eng:
        centers = np.random.default_rng(2).integers(M * eng.params.dop_lo, M * eng.params.dop_hi + 1, 32).astype(np.int32)
        calls = {"acq_search": lambda: eng.search(cap), "coherent_m4": lambda: eng.search_coherent(cap, M)}
        for hw in (4, 8):
            calls["aided_m4_hw%d" % hw] = (lambda hw=hw: eng.search_coherent_aided(cap, M, centers, hw))
        for fn in calls.values():
            for _ in range(5):
                fn()
        t = {k: [] for k in calls}
        for _ in range(steps):   # interleaved
            for k, fn in calls.items():
                t0 = time.perf_counter()
                fn()
                t[k].append((time.perf_counter() - t0) * 1e6)
        for k, v in t.items():
            res[k] = {"median_us": statistics.median(v), "min_us": min(v)}
    return res


def sensitivity(F, S, synth, torch, n_cap, cn0s):
    table = S.navstar()
    ms = (1, 4, 5)
    res = {"captures_per_point": n_cap, "centres": "true coherent index + seeded offset in [-M, M], half_width = 2M",
           "found": {}, "noise_snr_quantiles": {}}
    with F.AcqEngine(table, F.default_params(**CFG2)) as eng:
        for cn0 in cn0s:
            caps, tau, f = sensitivity_set(F, S, synth, torch, 1000 + int(cn0 * 10), n_cap, cn0)
            row = {}
            for m in ms:
                full = eng.search_coherent(caps, m, sel=[7])[:, 0]
                c = truth_centers(F, eng, m, f, int(cn0 * 10) + m)
                aided = eng.search_coherent_aided(caps, m, c.reshape(-1, 1), 2 * m, sel=[7])[:, 0]
                row["m%d" % m] = {"full": float(found(F, eng, full, m, tau, f).mean()),
                                  "aided": float(found(F, eng, aided, m, tau, f).mean())}
            res["found"][str(cn0)] = row
            print("cn0", cn0, row, flush=True)
        caps, _, _ = sensitivity_set(F, S, synth, torch, 99, 256, None)
        rng = np.random.default_rng(9)
        for m in ms:
            clo, chi = m * eng.params.dop_lo, m * eng.params.dop_hi
            for hw in (None, m, 2 * m, 4 * m):
                if hw is None:
                    snr = eng.search_coherent(caps, m)["snr"].reshape(-1)
                    W = eng.coherent_dops(m)
                else:
                    c = rng.integers(clo, chi + 1, (256, 32)).astype(np.int32)
                    snr = eng.search_coherent_aided(caps, m, c, hw)["snr"].reshape(-1)
                    W = 2 * hw + 1
                q = np.quantile(snr, [0.5, 0.99, 0.999])
                res["noise_snr_quantiles"]["m%d_w%d" % (m, W)] = {"m_coh": m, "cells_per_row": W, "rows": int(snr.size),
                                                                  "q50": float(q[0]), "q99": float(q[1]), "q999": float(q[2])}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tag", default="b200")
    ap.add_argument("--out", default="profiles")
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--sens-captures", type=int, default=128)
    args = ap.parse_args()
    import torch
    import flydog_sdr_gps_b200 as F
    from flydog_sdr_gps_b200 import sats as S
    from flydog_sdr_gps_b200 import synth
    out = {"gpu": gpu_info(), "l2_flushed": False,
           "note": "CUDA events; kernel times from the engine's profiling events; medians over --steps interleaved calls"}
    out["throughput_cfg2_128cap"] = throughput(F, S, synth, torch, args.steps)
    print(json.dumps(out["throughput_cfg2_128cap"]), flush=True)
    out["latency_k4_1cap_32prn_m4"] = latency(F, S, synth, 40 * args.steps)
    print(json.dumps(out["latency_k4_1cap_32prn_m4"]), flush=True)
    out["sensitivity_cfg2"] = sensitivity(F, S, synth, torch, args.sens_captures, [27.0, 29.0, 31.0])
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "coherent_aided_bench_%s.json" % args.tag)
    with open(path, "w") as fh:
        json.dump(out, fh, indent=1)
    print(json.dumps(out, indent=1))
    print("wrote", path)


if __name__ == "__main__":
    main()
