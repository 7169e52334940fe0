"""Peak-quality profile (acq_profile_device) at farm scale on one GPU.

Workload: the 1024-capture receiver farm (bench.farm_captures_numpy, 32 GPS PRNs), searched on the device path over the
full range (41 bins) and aided with W = 5 (centres by aided_bench.farm_centers).  For each search, CUDA events on one
non-default stream time these steps, interleaved on the same captures:
  search                  the search alone
  search_profile_det      the search + profile_device of the detected rows (ACQ_PROFILE_DETECTED), no lag profiles
  profile_all             k_profile alone, all 32768 rows, no lag profiles (behind a search of the same kind)
  profile_det             k_profile alone, detected rows only
  profile_all_vectors     k_profile alone, all rows, with the lag profiles (32768 x 4092 floats)
  profile_det_vectors     k_profile alone, detected rows, with the lag profiles
Also reported: evaluated rows; the bytes k_profile reads and writes, from shapes (K x (1 capture row + 1 code row) x
128 KiB per evaluated row, + L x 4 bytes of profile); and the distribution of ratio over the detected rows.

Records the GPU's name, power limit and maximum SM clock (nvidia-smi query) in the same run and writes
<out>/profile_bench_<tag>.json.  Usage: python tools/profile_bench.py --tag b200 [--out profiles] [--steps 20]
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

from aided_bench import farm_centers, gpu_info  # noqa: E402

ROW_BYTES = 16384 * 8   # one spectrum row: 16384 complex floats
THR = 16.0              # the engine's default C/A threshold (the farm's table is all C/A)
EXCL = 4


def run(F, S, torch, bench, steps):
    table = S.navstar()
    n_cap, n_sel, hw = bench.CAPTURES_TOTAL, 32, 2
    rows = n_cap * n_sel
    caps = bench.farm_captures_numpy(range(n_cap))
    centers = farm_centers(F, bench, n_cap, n_sel)
    res = {}
    with F.AcqEngine(table) as eng:
        K = eng.k_noncoh
        d_in = torch.from_numpy(caps.reshape(-1)).cuda()
        d_c = torch.from_numpy(centers.reshape(-1)).cuda()
        d_rec = torch.zeros(rows * 24, dtype=torch.uint8, device="cuda")
        d_pk = torch.zeros(rows * 16, dtype=torch.uint8, device="cuda")
        d_prof = torch.zeros(rows * F.LAGS_L1, dtype=torch.float32, device="cuda")
        # a non-default stream: its handle is non-NULL, so the engine launches on exactly this stream and the events
        # bracket its kernels (NULL would select the engine's own stream)
        st = torch.cuda.Stream()
        sp = st.cuda_stream
        torch.cuda.synchronize()
        searches = {"full_41": lambda: eng.search_device(d_in.data_ptr(), d_rec.data_ptr(), n_cap, stream_ptr=sp),
                    "aided_W5": lambda: eng.search_aided_device(d_in.data_ptr(), d_c.data_ptr(), hw, d_rec.data_ptr(), n_cap,
                                                                stream_ptr=sp)}

        def profile(det, vectors):
            eng.profile_device(d_rec.data_ptr(), d_pk.data_ptr(), rows, excl=EXCL, detected_only=det,
                               profile_dev=d_prof.data_ptr() if vectors else None, stream_ptr=sp)

        for kind, search in searches.items():
            arms = {"search": search,
                    "search_profile_det": lambda s=search: (s(), profile(True, False)),
                    "profile_all": lambda: profile(False, False),
                    "profile_det": lambda: profile(True, False),
                    "profile_all_vectors": lambda: profile(False, True),
                    "profile_det_vectors": lambda: profile(True, True)}
            for fn in arms.values():   # warm-up (a profile follows its own kind's search)
                for _ in range(2):
                    fn()
            torch.cuda.synchronize()
            ms = {k: [] for k in arms}
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
            for _ in range(steps):
                for k, fn in arms.items():   # interleaved on the same captures
                    ev[0].record(st)
                    fn()
                    ev[1].record(st)
                    ev[1].synchronize()
                    ms[k].append(ev[0].elapsed_time(ev[1]))
            search()
            profile(False, True)
            st.synchronize()
            rec = d_rec.cpu().numpy().view(F.RECORD_DTYPE).reshape(n_cap, n_sel)
            pk = d_pk.cpu().numpy().view(F.PEAK2_DTYPE).reshape(n_cap, n_sel)
            prof = d_prof.cpu().numpy().reshape(n_cap, n_sel, F.LAGS_L1)
            det = rec["snr"] >= THR
            n_det = int(det.sum())
            # the profile at the record's lag is the record's peak (bitwise), every row evaluated
            assert (pk["lag2"] >= 0).all()
            assert np.array_equal(np.take_along_axis(prof, rec["lag"][..., None], 2)[..., 0], rec["peak"])
            r = {"steps": steps}
            for k, v in ms.items():
                r[k] = {"median_ms": statistics.median(v), "min_ms": min(v), "max_ms": max(v)}
            r["rows"] = rows
            r["evaluated_rows"] = {"all": rows, "det": n_det}
            per_row = K * 2 * ROW_BYTES
            r["k_profile_read_bytes_per_row"] = per_row
            r["profile_write_bytes_per_row"] = F.LAGS_L1 * 4
            for m, n in (("all", rows), ("det", n_det)):
                t = r["profile_" + m]["median_ms"] * 1e-3
                tv = r["profile_%s_vectors" % m]["median_ms"] * 1e-3
                r["k_profile_us_per_row_" + m] = t * 1e6 / max(n, 1)
                r["k_profile_read_bytes_per_s_" + m] = n * per_row / t
                r["k_profile_bytes_per_s_%s_vectors" % m] = n * (per_row + F.LAGS_L1 * 4) / tv
            r["profile_det_over_search"] = (r["search_profile_det"]["median_ms"] - r["search"]["median_ms"]) / \
                r["search"]["median_ms"]
            ratio = pk["ratio"][det]
            r["ratio_detected_rows"] = {"min": float(ratio.min()), "p5": float(np.percentile(ratio, 5)),
                                        "median": float(np.median(ratio))}
            res[kind] = r
    res["l2"] = ("not flushed between steps: every step reads the same 1024 captures' spectra (128 MiB for K = 1) and the "
                 "32 satellites' code rows")
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--tag", default="b200")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"))
    ap.add_argument("--steps", type=int, default=20)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("profile_bench: no CUDA device (nothing is measured without one)")
    import bench
    import flydog_sdr_gps_b200 as F
    from flydog_sdr_gps_b200 import sats as S
    result = {"gpu": gpu_info(), "torch_gpu": torch.cuda.get_device_name(0), "farm": run(F, S, torch, bench, args.steps)}
    result["gpu_after"] = gpu_info()
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "profile_bench_%s.json" % args.tag)
    with open(path, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result))


if __name__ == "__main__":
    main()
