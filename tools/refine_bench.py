"""Device-resident refinement (acq_refine_device) at farm scale on one GPU.

Workload: the 1024-capture receiver farm (bench.farm_captures_numpy, 32 GPS PRNs), searched on the device path over the
full range (41 bins) and aided with W = 5 (centres by aided_bench.farm_centers).  For each search, CUDA events on one
non-default stream time these steps, interleaved on the same captures:
  search            the search alone
  search_refine_all the search + refine_device of all 32768 rows
  search_refine_det the search + refine_device of the detected rows only (ACQ_REFINE_DETECTED)
  refine_all        k_refine alone, all rows (behind a search of the same kind, whose spectra it reads)
  refine_det        k_refine alone, detected rows only
Also reported: refined rows; the bytes k_refine reads, from shapes (K x (1 capture row + 3 code rows) x 128 KiB per refined
row); and, for every injected signal the search detects, the median and p95 Doppler and code-phase errors of the refined
values (dop_hz, code_fs) next to those of the record's whole bin and whole /4 lag.

Records the GPU's name, power limit and maximum SM clock (nvidia-smi query) in the same run and writes
<out>/refine_bench_<tag>.json.  Usage: python tools/refine_bench.py --tag b200 [--out profiles] [--steps 20]
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


def errors(F, bench, rec, fine):
    """Errors against the injected values for every injected signal whose (capture, satellite) record is detected."""
    period = 4 * F.LAGS_L1   # code period in FS samples
    e = {"dop_fine": [], "dop_record": [], "code_fine": [], "code_record": []}

    def wrap(x):
        x = x % period
        return x - period if x > period / 2 else x
    for c in range(rec.shape[0]):
        for sat, tau, f, _, _ in bench.farm_signals(c):
            r, q = rec[c, sat], fine[c, sat]
            if not r["snr"] >= THR:
                continue
            e["dop_fine"].append(abs(float(q["dop_hz"]) - f))
            e["dop_record"].append(abs(float(r["dop"]) * F.BIN_HZ - f))
            e["code_fine"].append(abs(wrap(float(q["code_fs"]) - tau)))
            e["code_record"].append(abs(wrap(4.0 * float(r["lag"]) - tau)))
    out = {"signals_detected": len(e["dop_fine"])}
    for k, v in e.items():
        unit = "hz" if k.startswith("dop") else "fs_samples"
        out["%s_median_%s" % (k, unit)] = float(np.median(v))
        out["%s_p95_%s" % (k, unit)] = float(np.percentile(v, 95))
    return out


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
        d_fine = torch.zeros(rows * 16, dtype=torch.uint8, device="cuda")
        # a non-default stream: its handle is non-NULL, so the engine launches on exactly this stream and the events
        # bracket its kernels (NULL would select the engine's own stream)
        st = torch.cuda.Stream()
        sp = st.cuda_stream
        torch.cuda.synchronize()
        searches = {"full_41": lambda: eng.search_device(d_in.data_ptr(), d_rec.data_ptr(), n_cap, stream_ptr=sp),
                    "aided_W5": lambda: eng.search_aided_device(d_in.data_ptr(), d_c.data_ptr(), hw, d_rec.data_ptr(), n_cap,
                                                                stream_ptr=sp)}

        def refine(det):
            eng.refine_device(d_rec.data_ptr(), d_fine.data_ptr(), rows, detected_only=det, stream_ptr=sp)

        for kind, search in searches.items():
            arms = {"search": search,
                    "search_refine_all": lambda s=search: (s(), refine(False)),
                    "search_refine_det": lambda s=search: (s(), refine(True)),
                    "refine_all": lambda: refine(False),
                    "refine_det": lambda: refine(True)}
            for fn in arms.values():   # warm-up (the arms run in this order, so a refine follows its own kind's search)
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
            refine(False)
            st.synchronize()
            rec = d_rec.cpu().numpy().view(F.RECORD_DTYPE).reshape(n_cap, n_sel)
            fine = d_fine.cpu().numpy().view(F.FINE_DTYPE).reshape(n_cap, n_sel)
            refine(True)
            st.synchronize()
            fine_det = d_fine.cpu().numpy().view(F.FINE_DTYPE).reshape(n_cap, n_sel)
            n_det = int((rec["snr"] >= THR).sum())
            assert int((fine_det["ca_shift"] >= 0).sum()) == n_det and (fine["ca_shift"] >= 0).all()
            r = {"steps": steps}
            for k, v in ms.items():
                r[k] = {"median_ms": statistics.median(v), "min_ms": min(v), "max_ms": max(v)}
            r["rows"] = rows
            r["refined_rows"] = {"all": rows, "det": n_det}
            per_row = K * 4 * ROW_BYTES
            r["k_refine_bytes"] = {"all": rows * per_row, "det": n_det * per_row, "per_refined_row": per_row}
            for m in ("all", "det"):
                t = r["refine_" + m]["median_ms"] * 1e-3
                r["k_refine_bytes_per_s_" + m] = r["k_refine_bytes"][m] / t
                r["k_refine_us_per_refined_row_" + m] = t * 1e6 / max(r["refined_rows"][m], 1)
                r["refine_over_search_" + m] = (r["search_refine_" + m]["median_ms"] - r["search"]["median_ms"]) / \
                    r["search"]["median_ms"]
            r["accuracy"] = errors(F, bench, rec, fine)
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
        sys.exit("refine_bench: no CUDA device (nothing is measured without one)")
    import bench
    import flydog_sdr_gps_b200 as F
    from flydog_sdr_gps_b200 import sats as S
    result = {"gpu": gpu_info(), "torch_gpu": torch.cuda.get_device_name(0), "farm": run(F, S, torch, bench, args.steps)}
    result["gpu_after"] = gpu_info()
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "refine_bench_%s.json" % args.tag)
    with open(path, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result))


if __name__ == "__main__":
    main()
