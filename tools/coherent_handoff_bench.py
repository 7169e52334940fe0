"""Hand-off of coherent records (acq_refine_coherent_device, acq_profile_coherent_device) on one GPU: cost, accuracy,
peak quality.

  cost      the cfg2 shape of tools/coherent_bench.py (CFG2: K = 20, half-bins, +-80), 128 captures x 32 PRN through the
            device forms at M = 1, 4 and 5: CUDA events on a non-default stream around the coherent search, around
            k_refine_coh and around k_profile_coh (no lag profiles) over all 4096 rows, and over the rows with snr >= the
            noise-only 99.9 % snr quantile of that M (profiles/coherent_bench_b200.json) -- each against the search's
            own time in the same run.  Medians over --steps interleaved calls.
  accuracy  sensitivity_set's captures (one PRN at a random code phase that is a multiple of 4 samples, so on a lag, and
            a Doppler uniform in +-9 kHz) at 31 and 35 dB-Hz, M = 1, 4, 5: median and p95 of the refined Doppler and
            code-phase errors against the injected truth over the found rows (coherent_bench.found), beside the grid-only
            figures (h BIN / F, 4 lag).  The same with code phases at any sample (handoff_set), where the grid's code
            error is not zero.
  quality   acq_peak2.ratio quantiles (5 / 50 / 95 %) of the noise-only rows of sensitivity_set (128 captures x 32 PRN)
            against the found signal rows at 31 and 35 dB-Hz, per M.

Records the GPU's name, power limit and maximum SM clock (nvidia-smi query) in the same run and writes
<out>/coherent_handoff_bench_<tag>.json.  Usage: python tools/coherent_handoff_bench.py --tag b200 [--out profiles]
"""
import argparse
import json
import os
import statistics
import sys

import numpy as np

TOOLS = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(TOOLS)
sys.path.insert(0, ROOT)
sys.path.insert(0, TOOLS)

from aided_bench import gpu_info  # noqa: E402
from coherent_bench import CFG2, found, sensitivity_set  # noqa: E402

MS = (1, 4, 5)
CODE_PERIOD_FS = 4 * 4092   # FS samples of one C/A code period


def handoff_set(F, S, synth, torch, seed, n_cap, cn0, sat=7, K=20):
    """sensitivity_set with the code phase at any FS sample (tau uniform in 0..16367), so the truth lies between lags."""
    rng = np.random.default_rng(seed)
    tau = rng.integers(0, CODE_PERIOD_FS, n_cap)
    f = rng.uniform(-9000.0, 9000.0, n_cap)
    sig = [[(sat, int(tau[c]), float(f[c]), float(cn0), float(rng.uniform(0, 2 * np.pi)))] for c in range(n_cap)]
    caps = synth.make_capture_batch_torch([seed * 100_000 + c for c in range(n_cap)], K, S.navstar(), sig, "cuda")
    return caps.cpu().numpy(), tau, f


def _wrap(x, period):
    return (np.asarray(x, np.float64) + period / 2) % period - period / 2


def _stats(e):
    e = np.abs(np.asarray(e, np.float64))
    if e.size == 0:
        return {"n": 0}
    return {"n": int(e.size), "median": float(np.median(e)), "p95": float(np.quantile(e, 0.95))}


def accuracy(F, eng, rec, fine, m_coh, tau, f_hz):
    """Errors of the refined and the grid-only Doppler (Hz) and code phase (FS samples) over the found rows."""
    ok = found(F, eng, rec, m_coh, tau, f_hz)
    tau, f_hz = np.asarray(tau)[ok], np.asarray(f_hz)[ok]
    r, g = rec[ok], fine[ok]
    return {"found": float(ok.mean()),
            "dop_hz_refined": _stats(g["dop_hz"] - f_hz),
            "dop_hz_grid": _stats(eng.coherent_dop_hz(r["dop"], m_coh) - f_hz),
            "code_fs_refined": _stats(_wrap(g["code_fs"] - tau, CODE_PERIOD_FS)),
            "code_fs_grid": _stats(_wrap(4.0 * r["lag"] - tau, CODE_PERIOD_FS))}


def _thresholds():
    """Noise-only 99.9 % snr quantile per M of the coherent search on this workload (tools/coherent_bench.py's run)."""
    with open(os.path.join(ROOT, "profiles", "coherent_bench_b200.json")) as fh:
        q = json.load(fh)["sensitivity_cfg2"]["noise_snr_quantiles"]
    return {m: q["m%d" % m]["q999"] for m in MS}


def cost(F, S, synth, torch, steps):
    table = S.navstar()
    n_cap, n_sel = 128, 32
    n = n_cap * n_sel
    caps, _, _ = sensitivity_set(F, S, synth, torch, 5, n_cap, 30.0)
    thr = _thresholds()
    res = {"rows": n, "min_snr_thresholds": {str(m): thr[m] for m in MS}}
    with F.AcqEngine(table, F.default_params(**CFG2)) as eng:
        d_in = torch.from_numpy(caps.reshape(-1)).cuda()
        d_rec = torch.zeros(n * 24, dtype=torch.uint8, device="cuda")
        d_fine = torch.zeros(n * 16, dtype=torch.uint8, device="cuda")
        d_pk = torch.zeros(n * 16, dtype=torch.uint8, device="cuda")
        st = torch.cuda.Stream()
        sp = st.cuda_stream
        torch.cuda.synchronize()

        def timed(fn):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(st)
            fn()
            b.record(st)
            b.synchronize()
            return a.elapsed_time(b)

        for m in MS:
            calls = {
                "search": lambda: eng.search_coherent_device(d_in.data_ptr(), m, d_rec.data_ptr(), n_cap, stream_ptr=sp),
                "refine_all": lambda: eng.refine_coherent_device(d_rec.data_ptr(), d_fine.data_ptr(), n, stream_ptr=sp),
                "profile_all": lambda: eng.profile_coherent_device(d_rec.data_ptr(), d_pk.data_ptr(), n, stream_ptr=sp),
                "refine_above_thr": lambda: eng.refine_coherent_device(d_rec.data_ptr(), d_fine.data_ptr(), n,
                                                                       min_snr=thr[m], stream_ptr=sp),
                "profile_above_thr": lambda: eng.profile_coherent_device(d_rec.data_ptr(), d_pk.data_ptr(), n,
                                                                         min_snr=thr[m], stream_ptr=sp),
            }
            for fn in calls.values():   # warm-up (the search first: the hand-off reads its spectra)
                fn()
            torch.cuda.synchronize()
            t = {k: [] for k in calls}
            for _ in range(steps):
                for k, fn in calls.items():
                    t[k].append(timed(fn))
            rec = d_rec.cpu().numpy().view(F.RECORD_DTYPE)
            r = {k: {"median_ms": statistics.median(v), "min_ms": min(v)} for k, v in t.items()}
            r["rows_above_thr"] = int((rec["snr"] >= thr[m]).sum())
            for k in calls:
                if k != "search":
                    r[k]["vs_search"] = r[k]["median_ms"] / r["search"]["median_ms"]
            res["m%d" % m] = r
            print("cost M = %d" % m, json.dumps(r), flush=True)
    return res


def accuracy_and_quality(F, S, synth, torch, n_cap):
    table = S.navstar()
    res = {"captures_per_point": n_cap, "accuracy_on_lag_code": {}, "accuracy_any_code": {}, "ratio": {}}
    with F.AcqEngine(table, F.default_params(**CFG2)) as eng:
        sig_ratio = {m: [] for m in MS}
        for cn0 in (31.0, 35.0):
            for key, maker in (("accuracy_on_lag_code", sensitivity_set), ("accuracy_any_code", handoff_set)):
                caps, tau, f = maker(F, S, synth, torch, 2000 + int(cn0 * 10), n_cap, cn0)
                res[key][str(cn0)] = {}
                for m in MS:
                    rec = eng.search_coherent(caps, m, sel=[7])
                    fine = eng.refine_coherent(rec)[:, 0]
                    res[key][str(cn0)]["m%d" % m] = accuracy(F, eng, rec[:, 0], fine, m, tau, f)
                    if key == "accuracy_on_lag_code":
                        ok = found(F, eng, rec[:, 0], m, tau, f)
                        sig_ratio[m].append(eng.profile_coherent(rec)[:, 0]["ratio"][ok])
                print(key, cn0, json.dumps(res[key][str(cn0)]), flush=True)
        caps, _, _ = sensitivity_set(F, S, synth, torch, 99, n_cap, None)
        for m in MS:
            rec = eng.search_coherent(caps, m)
            noise = eng.profile_coherent(rec)["ratio"].reshape(-1)
            sig = np.concatenate(sig_ratio[m])
            res["ratio"]["m%d" % m] = {
                "noise_rows": int(noise.size), "signal_rows": int(sig.size),
                "noise_q05_q50_q95": [float(x) for x in np.quantile(noise, [0.05, 0.5, 0.95])],
                "noise_max": float(noise.max()),
                "signal_q05_q50_q95": [float(x) for x in np.quantile(sig, [0.05, 0.5, 0.95])] if sig.size else None}
            print("ratio M = %d" % m, json.dumps(res["ratio"]["m%d" % m]), flush=True)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tag", default="b200")
    ap.add_argument("--out", default="profiles")
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--captures", type=int, default=128)
    args = ap.parse_args()
    import torch
    import flydog_sdr_gps_b200 as F
    from flydog_sdr_gps_b200 import sats as S
    from flydog_sdr_gps_b200 import synth
    out = {"gpu": gpu_info(), "note": "CUDA events on a non-default stream; medians over --steps interleaved calls"}
    out["cost_cfg2_128cap_32prn"] = cost(F, S, synth, torch, args.steps)
    out.update(accuracy_and_quality(F, S, synth, torch, args.captures))
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "coherent_handoff_bench_%s.json" % args.tag)
    with open(path, "w") as fh:
        json.dump(out, fh, indent=1)
    print(json.dumps(out, indent=1))
    print("wrote", path)


if __name__ == "__main__":
    main()
