"""Coherent integration across capture blocks (acq_search_coherent) on one GPU: latency, throughput, sensitivity.

  latency      one capture, 32 GPS PRNs, a K = 4 engine (full bins, +-20): per-call time of acq_search against
               acq_search_coherent at M = 1, 2 and 4 (host clock around the synchronous calls, after warm-up).
  throughput   a cfg2-shaped engine (K = 20, half-bins, +-80) over 128 captures through the device forms, at M = 1, 2, 4
               and 5 against acq_search_device: search-kernel time (the engine's own CUDA events around the search
               launch, acq_set_profiling) and the whole search (CUDA events on a non-default stream), block-IFFTs per
               second (captures x 32 x cells x K over the search-kernel time), and the time per block-IFFT of
               k_search_l1_coh over that of k_search_l1_multi.  The capture spectra of one search (2560 blocks x F
               variants x 128 KiB) exceed the 126 MB L2 at every M, so L2 is not flushed between calls.
  sensitivity  the same engine and 20-block bytes searched at M = 1, 4 and 5: found rate (lag within +-1 of the true
               code phase, Doppler within one coherent step of the truth) against C/N0, one PRN per capture at a random
               code phase and Doppler; and the snr quantiles (50 / 99 / 99.9 %) of noise-only captures per M, from which a
               threshold for each M can be chosen.

Records the GPU's name, power limit and maximum SM clock (nvidia-smi query) in the same run and writes
<out>/coherent_bench_<tag>.json.  Usage: python tools/coherent_bench.py --tag b200 [--out profiles] [--steps 20]
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

CFG2 = dict(dop_lo=-80, dop_hi=80, half_bin=1, k_noncoh=20, thr_l1=2.6)


def found(F, eng, rec, m_coh, tau, f_hz):
    """lag within +-1 (circular, L = 4092) of tau / 4 and Doppler within one coherent step (BIN_HZ / F) of f_hz."""
    dl = np.abs(rec["lag"] - np.round(np.asarray(tau) / 4.0).astype(np.int64) % F.LAGS_L1)
    dl = np.minimum(dl, F.LAGS_L1 - dl)
    step = F.BIN_HZ / (m_coh * (1 + eng.params.half_bin))
    return (dl <= 1) & (np.abs(eng.coherent_dop_hz(rec["dop"], m_coh) - f_hz) <= step)


def sensitivity_set(F, S, synth, torch, seed, n_cap, cn0, sat=7, K=20):
    """n_cap captures of K blocks with one PRN (sat) at C/N0 cn0 (None: noise only): random code phase (a multiple of 4
    samples) and Doppler uniform in +-9 kHz.  Returns (bytes uint8 [n_cap, K*8192], tau, f_hz)."""
    rng = np.random.default_rng(seed)
    tau = 4 * rng.integers(0, 4092, n_cap)
    f = rng.uniform(-9000.0, 9000.0, n_cap)
    sig = [[] if cn0 is None else [(sat, int(tau[c]), float(f[c]), float(cn0), float(rng.uniform(0, 2 * np.pi)))]
           for c in range(n_cap)]
    caps = synth.make_capture_batch_torch([seed * 100_000 + c for c in range(n_cap)], K, S.navstar(), sig, "cuda")
    return caps.cpu().numpy(), tau, f


def latency(F, S, synth, steps):
    table = S.navstar()
    cap = np.ascontiguousarray(synth.make_capture(4711, 4, table, [(3, 4000, 3.4 * F.BIN_HZ, 44, 0.5)]))
    res = {}
    with F.AcqEngine(table, F.default_params(k_noncoh=4)) as eng:
        calls = {"acq_search": lambda: eng.search(cap)}
        for m in (1, 2, 4):
            calls["coherent_m%d" % m] = (lambda m=m: eng.search_coherent(cap, m))
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
        torch.cuda.synchronize()
        calls = {"acq_search_device": (lambda: eng.search_device(d_in.data_ptr(), d_rec.data_ptr(), n_cap, stream_ptr=sp),
                                       eng.n_dop)}
        for m in (1, 2, 4, 5):
            calls["coherent_m%d" % m] = ((lambda m=m: eng.search_coherent_device(d_in.data_ptr(), m, d_rec.data_ptr(),
                                                                                  n_cap, stream_ptr=sp)),
                                         eng.coherent_dops(m))
        kern = {k: [] for k in calls}
        whole = {k: [] for k in calls}
        for k, (fn, _) in calls.items():
            fn()
        torch.cuda.synchronize()
        for _ in range(steps):
            for k, (fn, _) in calls.items():   # interleaved; kernel times from the engine's events (profiling on)
                eng.set_profiling(True)
                fn()
                kern[k].append(eng.kernel_ms()["search"])
                eng.set_profiling(False)
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(st)
                fn()
                b.record(st)
                b.synchronize()
                whole[k].append(a.elapsed_time(b))
        for k, (_, n_dop) in calls.items():
            ms = statistics.median(kern[k])
            n_ifft = n_cap * n_sel * n_dop * K
            res[k] = {"cells_per_row": n_dop, "search_kernel_ms": ms, "search_kernel_ms_min": min(kern[k]),
                      "whole_search_ms": statistics.median(whole[k]), "block_iffts": n_ifft,
                      "block_iffts_per_s": n_ifft / (ms * 1e-3)}
        base = res["acq_search_device"]["search_kernel_ms"] / res["acq_search_device"]["block_iffts"]
        for k in calls:
            res[k]["time_per_block_ifft_vs_l1_multi"] = res[k]["search_kernel_ms"] / res[k]["block_iffts"] / base
    return res


def sensitivity(F, S, synth, torch, n_cap, cn0s):
    table = S.navstar()
    ms = (1, 4, 5)
    res = {"captures_per_point": n_cap, "found": {}, "noise_snr_quantiles": {}}
    with F.AcqEngine(table, F.default_params(**CFG2)) as eng:
        for cn0 in cn0s:
            caps, tau, f = sensitivity_set(F, S, synth, torch, 1000 + int(cn0 * 10), n_cap, cn0)
            res["found"][str(cn0)] = {("m%d" % m): float(found(F, eng, eng.search_coherent(caps, m, sel=[7])[:, 0], m, tau, f).mean())
                                      for m in ms}
            print("cn0", cn0, res["found"][str(cn0)], flush=True)
        caps, _, _ = sensitivity_set(F, S, synth, torch, 99, 256, None)
        for m in (1, 2, 4, 5):
            snr = eng.search_coherent(caps, m)["snr"].reshape(-1)
            q = np.quantile(snr, [0.5, 0.99, 0.999])
            res["noise_snr_quantiles"]["m%d" % m] = {"rows": int(snr.size), "q50": float(q[0]), "q99": float(q[1]),
                                                     "q999": float(q[2])}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tag", default="b200")
    ap.add_argument("--out", default="profiles")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--sens-captures", type=int, default=128)
    args = ap.parse_args()
    import torch
    import flydog_sdr_gps_b200 as F
    from flydog_sdr_gps_b200 import sats as S
    from flydog_sdr_gps_b200 import synth
    out = {"gpu": gpu_info(), "l2_flushed": False,
           "note": "CUDA events; kernel times from the engine's profiling events; medians over --steps interleaved calls"}
    out["latency_k4_1cap_32prn"] = latency(F, S, synth, 10 * args.steps)
    print(json.dumps(out["latency_k4_1cap_32prn"]), flush=True)
    out["throughput_cfg2_128cap"] = throughput(F, S, synth, torch, args.steps)
    print(json.dumps(out["throughput_cfg2_128cap"]), flush=True)
    out["sensitivity_cfg2"] = sensitivity(F, S, synth, torch, args.sens_captures, [23.0, 25.0, 27.0, 29.0, 31.0])
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "coherent_bench_%s.json" % args.tag)
    with open(path, "w") as fh:
        json.dump(out, fh, indent=1)
    print(json.dumps(out, indent=1))
    print("wrote", path)


if __name__ == "__main__":
    main()
