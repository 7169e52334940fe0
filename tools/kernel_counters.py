#!/usr/bin/env python3
"""profiles/r2_kernel_counters.json: per-tile ncu counters of the search kernels, read by bench.py for
roofline.traffic and roofline.frac_pipe_measured.  Input: the summaries tools/ncu_summary.py wrote under profiles/.
    python tools/kernel_counters.py"""
import json
import os

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# (config, summary file, tiles of the captured launch, what ran)
CAPTURES = [
    ("cfg5", "r2_ncu_l1_k1_cfg5.json", 128 * 32 * 41, "k_search_l1_cr, 128 captures x 32 PRNs x 41 bins (tools/ncu_driver.py cfg5 128)"),
    ("cfg1", "r2_ncu_l1_k1_cfg1.json", 32 * 41, "k_search_l1_cr on the static stride, one capture x 32 PRNs x 41 bins"),
    ("cfg2", "r2_ncu_l1_multi_cfg2.json", 32 * 161 * 20, "k_search_l1_multi, 32 PRNs x 161 half-bins x K = 20"),
    ("cfg3", "r2_ncu_e1b_cfg3.json", 50 * 81, "k_search_e1b, 50 PRNs x 81 bins"),
    ("cfg3_k4", "r2_ncu_e1b_multi_cfg3k4.json", 50 * 81 * 4, "k_search_e1b_multi, 50 PRNs x 81 bins x K = 4"),
]
SCALE = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}


def val(d, key):
    v, unit = d[key]
    return float(str(v).replace(",", "")) * SCALE.get(unit, 1.0)


def main():
    out = {"_doc": "per-tile counters of ONE launch of each search kernel under `ncu --set full --clock-control none` "
                   "(a tile = one inverse FFT of one (sat, Doppler, block)); dram bytes are cold-cache (ncu flushes "
                   "between replay passes)."}
    for cfg, name, tiles, what in CAPTURES:
        path = os.path.join(ROOT, "profiles", name)
        if not os.path.exists(path):
            continue
        d = json.load(open(path))
        out[cfg] = {
            "kernel": d["Kernel Name"][0], "what": what, "tiles": tiles, "profile": "profiles/" + name,
            "duration_ms_under_ncu": val(d, "gpu__time_duration.sum") * (1e-3 if d["gpu__time_duration.sum"][1] == "us" else 1.0),
            "smem_wavefronts_per_tile": val(d, "l1tex__data_pipe_lsu_wavefronts_mem_shared.sum") / tiles,
            "smem_store_conflict_wavefronts_per_tile": val(d, "l1tex__data_bank_conflicts_pipe_lsu_mem_shared_op_st.sum") / tiles,
            "dram_bytes_per_tile": (val(d, "dram__bytes_read.sum") + val(d, "dram__bytes_write.sum")) / tiles,
            "lsu_pipe_pct": val(d, "l1tex__data_pipe_lsu_wavefronts.avg.pct_of_peak_sustained_elapsed"),
            "fma_pipe_pct": val(d, "sm__pipe_fma_cycles_active.avg.pct_of_peak_sustained_active"),
            "issue_active_pct": val(d, "smsp__issue_active.avg.pct_of_peak_sustained_active"),
            "registers": int(val(d, "launch__registers_per_thread")),
        }
    out["cfg4"] = {"note": "cfg4 runs k_search_l1_cr (cfg1's) and k_search_e1b (cfg3's) back to back"}
    json.dump(out, open(os.path.join(ROOT, "profiles", "r2_kernel_counters.json"), "w"), indent=1, sort_keys=True)
    for k, v in out.items():
        if isinstance(v, dict) and "tiles" in v:
            print(k, {a: (round(b, 2) if isinstance(b, float) else b) for a, b in v.items() if a not in ("what", "profile", "kernel")})


if __name__ == "__main__":
    main()
