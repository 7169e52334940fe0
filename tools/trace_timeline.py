#!/usr/bin/env python3
"""Timeline of ONE search from the "trace" variant library (%globaltimer stamps of every CTA: entry, after the wait
for the preceding grid, exit).  Run on the GPU box:
    python tools/trace_timeline.py cfg1 [cfg4 ...]        -> one summary line per kernel, times in us from the first stamp"""
import ctypes as C
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import flydog_sdr_gps_b200 as F
from flydog_sdr_gps_b200 import _lib, scenarios, synth

NAMES = ["front_end", "fwd_fft", "search_l1", "search_e1b", "pick", "e1b_cluster"]
VARIANT = os.environ.get("TRACE_VARIANT", "trace")
L = _lib.load_variant(VARIANT)
L.acq_trace_read.argtypes = [C.c_void_p, C.c_int]
total = L.acq_trace_read(None, 0)
buf = np.zeros(total, np.uint64)

for cfg in sys.argv[1:] or ["cfg1"]:
    table = scenarios.table(cfg)
    kw = scenarios.params_kw(cfg)
    ncap = int(os.environ.get("TRACE_CAPS", "1"))
    cap = np.concatenate([synth.make_capture(1 + i, kw.get("k_noncoh", 1), table, scenarios.signals(cfg, 1 + i)) for i in range(ncap)])
    with F.AcqEngine(table, F.default_params(**kw), variant=VARIANT) as eng:
        import time
        for _ in range(20):
            eng.search(cap)
        L.acq_trace_read(buf.ctypes.data, total)
        if os.environ.get("TRACE_FLUSH"):   # cold L2, as between the bench's timed steps: a 256 MiB fill
            import torch
            torch.empty(256 << 20, dtype=torch.uint8, device="cuda").fill_(1)
            torch.cuda.synchronize()
        t0 = time.perf_counter()
        eng.search(cap)
        host_us = (time.perf_counter() - t0) * 1e6
        L.acq_trace_read(buf.ctypes.data, total)
    tr = buf.reshape(len(NAMES), -1, 4).astype(np.int64)
    start = tr[tr > 0].min()
    print("== %s: host acq_search() %.1f us" % (cfg, host_us))
    for k, name in enumerate(NAMES):
        used = tr[k][:, 0] > 0
        if not used.any():
            continue
        e, w, x = [(tr[k][used][:, s] - start) / 1e3 for s in range(3)]
        x = x[tr[k][used][:, 2] > 0] if (tr[k][used][:, 2] > 0).any() else np.array([np.nan])
        w = w[tr[k][used][:, 1] > 0] if (tr[k][used][:, 1] > 0).any() else np.array([np.nan])
        extra = ""
        if (tr[k][used][:, 3] > 0).any():
            extra = "  mark3 %6.1f" % ((tr[k][used][:, 3].max() - start) / 1e3)
        if os.environ.get("TRACE_DUMP") and name.startswith("search"):
            xs = np.sort(x)
            print("  %s exit deciles:" % name, " ".join("%.1f" % v for v in np.percentile(xs, range(0, 101, 10))))
            ex_all = (tr[k][used][:, 2] - start) / 1e3
            print("  %s exit by CTA index (every 8th):" % name, " ".join("%.0f" % v for v in ex_all[::8]))
            m3 = (tr[k][used][:, 3] - start) / 1e3
            if (tr[k][used][:, 3] > 0).any():
                print("  %s mark3 by CTA index (every 8th):" % name, " ".join("%.0f" % v for v in m3[::8]))
            print("  %s past-wait by CTA index (every 8th):" % name, " ".join("%.1f" % v for v in ((tr[k][used][:, 1] - start) / 1e3)[::8]))
        if name == "fwd_fft" and (tr[k][64:320, 3] > 0).any():   # cluster forward FFT: inner stamps of thread 0
            for lbl, off in (("loads arrived", 64), ("sub-FFT done", 128), ("cluster barrier passed", 192), ("combine + stores issued", 256)):
                v = tr[k][off:off + 64, 3]
                v = (v[v > 0] - start) / 1e3
                print("  fwd_fft %-24s %6.2f..%6.2f" % (lbl, v.min(), v.max()))
        print("  %-12s ctas %4d  entry %6.1f..%6.1f  past-wait %6.1f..%6.1f  exit %6.1f..%6.1f (median %6.1f)%s" % (
            name, used.sum(), e.min(), e.max(), w.min(), w.max(), x.min(), x.max(), np.median(x), extra))
