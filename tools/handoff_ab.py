#!/usr/bin/env python3
"""Byte A/B of the hand-off kernels between two builds of the library (GPU): refine / refine_device (all rows and
detected only) and profile / profile_device (with lag vectors) after the searches of test_gpu_profile.SHAPES and an aided
search, and the four coherent forms after coherent searches at M = 1..5 on full and half bins, full and aided.
    python tools/handoff_ab.py run OUT.npz            (ACQ_B200_LIB selects the library)
    python tools/handoff_ab.py compare A.npz B.npz    (exit 1 unless every output is byte-equal)"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def handoff(F, eng, rec, n_prof, coherent, out, key):
    """Every hand-off output of the records `rec` of the engine's last search, as raw bytes under `key`."""
    import torch
    n = rec.size
    d_rec = torch.from_numpy(np.ascontiguousarray(rec).reshape(-1).view(np.uint8).copy()).cuda()
    new = lambda nbytes: torch.zeros(max(int(nbytes), 1), dtype=torch.uint8, device="cuda")
    host = lambda t: t.cpu().numpy()
    if coherent:
        out[key + "/refine"] = eng.refine_coherent(rec)
        out[key + "/profile"], out[key + "/lags"] = eng.profile_coherent(rec, want_profile=True)
    else:
        out[key + "/refine"] = eng.refine(rec)
        out[key + "/profile"], out[key + "/lags"] = eng.profile(rec, want_profile=True)
    thr = float(np.median(rec["snr"]))
    for sub in ("all", "detected"):
        d_f, d_p, d_q = new(n * 16), new(n * 16), new(n_prof * 4)
        torch.cuda.synchronize()
        if coherent:
            min_snr = thr if sub == "detected" else 0.0
            eng.refine_coherent_device(d_rec.data_ptr(), d_f.data_ptr(), n, min_snr=min_snr)
            eng.profile_coherent_device(d_rec.data_ptr(), d_p.data_ptr(), n, min_snr=min_snr, profile_dev=d_q.data_ptr())
        else:
            eng.refine_device(d_rec.data_ptr(), d_f.data_ptr(), n, detected_only=sub == "detected")
            eng.profile_device(d_rec.data_ptr(), d_p.data_ptr(), n, detected_only=sub == "detected",
                               profile_dev=d_q.data_ptr())
        torch.cuda.synchronize()
        out["%s/refine_device_%s" % (key, sub)] = host(d_f)
        out["%s/profile_device_%s" % (key, sub)] = host(d_p)
        out["%s/lags_device_%s" % (key, sub)] = host(d_q)


def run(path):
    import flydog_sdr_gps_b200 as F
    from flydog_sdr_gps_b200 import sats as S, synth
    from test_gpu_profile import SHAPES, _shape
    out = {}
    for name in SHAPES:
        table, kw, cap, sel = _shape(name)
        with F.AcqEngine(table, F.default_params(**kw)) as eng:
            rec = eng.search(cap, sel=sel)
            n_prof = int(eng.profile_offsets(rec.shape[0], sel)[-1])
            handoff(F, eng, rec, n_prof, False, out, name)
            if name == "cfg1":   # aided: each row's window around its record's Doppler
                rec = eng.search_aided(cap, rec["dop"] + 2, 3, sel=sel)
                handoff(F, eng, rec, n_prof, False, out, "cfg1_aided")
    nav = S.navstar()
    sel = np.array([9, 14, 3, 22], np.int32)
    for M in range(1, 6):
        for hb in (0, 1):
            Fv = M * (1 + hb)
            K = 2 * M
            sig = [(9, 3003, (2 * Fv + 1.3) / Fv * F.BIN_HZ, 42, 0.9), (3, 12000, -3.4 * F.BIN_HZ, 43, 2.1)]
            cap = synth.make_capture(600 + 10 * M + hb, K, nav, sig)
            kw = dict(k_noncoh=K, half_bin=hb, dop_lo=-5 * (1 + hb), dop_hi=4 * (1 + hb))
            with F.AcqEngine(nav, F.default_params(**kw)) as eng:
                rec = eng.search_coherent(cap, M, sel=sel)
                handoff(F, eng, rec, rec.size * F.LAGS_L1, True, out, "coh_m%d_hb%d" % (M, hb))
                rec = eng.search_coherent_aided(cap, M, rec["dop"] - 1, 2 * M, sel=sel)
                handoff(F, eng, rec, rec.size * F.LAGS_L1, True, out, "coh_aided_m%d_hb%d" % (M, hb))
    np.savez(path, **{k: np.ascontiguousarray(v).reshape(-1).view(np.uint8) for k, v in out.items()})
    print("wrote", len(out), "outputs to", path)


def compare(a, b):
    A, B = np.load(a), np.load(b)
    bad = sorted(set(A.files) ^ set(B.files)) + [k for k in sorted(set(A.files) & set(B.files)) if A[k].tobytes() != B[k].tobytes()]
    print("%d outputs, %d differ%s" % (len(A.files), len(bad), (": " + ", ".join(bad)) if bad else ""))
    return not bad


if __name__ == "__main__":
    if sys.argv[1] == "run":
        run(sys.argv[2])
    else:
        sys.exit(0 if compare(sys.argv[2], sys.argv[3]) else 1)
