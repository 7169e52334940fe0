#!/usr/bin/env python3
"""Bitwise A/B of a variant library against the product on K = 1 C/A searches of several shapes (GPU).
    python tools/ab_equal.py l1_cta"""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import flydog_sdr_gps_b200 as F
from flydog_sdr_gps_b200 import sats as S, scenarios, synth

variant = sys.argv[1]
table = S.navstar()
cap = synth.make_capture(3, 1, table, scenarios.signals("cfg1", 3))
cap2 = synth.make_capture(5, 1, table, scenarios.signals("cfg1", 5))
ok = True
for kw, caps, sel in (({}, [cap], None), ({}, [cap, cap2] * 20, None), (dict(dop_lo=-3, dop_hi=1), [cap2], np.array([2], np.int32)),
                      (dict(dop_lo=0, dop_hi=0), [cap], np.array([6], np.int32)), (dict(dop_lo=-20, dop_hi=20), [cap2, cap], np.array([2, 6, 10, 13, 18], np.int32))):
    out = {}
    for kind, v in (("product", None), ("variant", variant)):
        with F.AcqEngine(table, F.default_params(**kw), variant=v) as eng:
            out[kind] = eng.search(np.concatenate(caps), sel=sel, want_grid=True)
    (ra, ga), (rb, gb) = out["product"], out["variant"]
    same = all(np.array_equal(ga[f], gb[f]) for f in ("peak", "lag", "noise", "snr")) and ra.tobytes() == rb.tobytes()
    print(kw, len(caps), "captures", "sel", None if sel is None else len(sel), "bitwise equal:", same)
    ok &= same
sys.exit(0 if ok else 1)
