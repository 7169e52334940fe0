#!/usr/bin/env python3
"""Host-side latency of acq_search() (C ABI, host buffers) for single-capture searches, per library variant.
    python tools/e2e_latency.py [variant|product ...]     (configs cfg1 cfg4 cfg3, and one satellite = the literal SearchTask step)
    E2E_CAPS=2,4: additionally cfg1 searches of that many captures per call (where k_search_l1_cr starts claiming chunks of tiles)"""
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import flydog_sdr_gps_b200 as F
from flydog_sdr_gps_b200 import scenarios, synth

CAPS = [int(x) for x in os.environ.get("E2E_CAPS", "").split(",") if x]
for variant in sys.argv[1:] or ["product"]:
    for cfg, sel, ncap in [("cfg1", None, 1), ("cfg1", np.array([7], np.int32), 1), ("cfg4", None, 1), ("cfg3", None, 1)] + [("cfg1", None, n) for n in CAPS]:
        table = scenarios.table(cfg)
        kw = scenarios.params_kw(cfg)
        cap = np.concatenate([synth.make_capture(1 + i, 1, table, scenarios.signals(cfg, 1 + i)) for i in range(ncap)])
        with F.AcqEngine(table, F.default_params(**kw), variant=None if variant == "product" else variant) as eng:
            n_sel = len(table) if sel is None else len(sel)
            out = np.zeros(n_sel * ncap, F.RECORD_DTYPE)
            for _ in range(50):
                eng.search_ptr(cap.ctypes.data, ncap, out.ctypes.data, sel=sel)
            ts = []
            for _ in range(1000):
                t0 = time.perf_counter()
                eng.search_ptr(cap.ctypes.data, ncap, out.ctypes.data, sel=sel)
                ts.append(time.perf_counter() - t0)
            ts = np.array(ts) * 1e6
            print("%-8s %s %-9s acq_search median %.1f us  p10 %.1f  min %.1f" % (
                variant, cfg, ("all" if sel is None else "1 sat") + ("" if ncap == 1 else " x%d" % ncap), np.median(ts), np.percentile(ts, 10), ts.min()), flush=True)
