"""GPU suite (-m gpu) of the precision tier: every non-coherent search kernel's cells, records, lag profiles,
second-peak rows and refinements (k_refine) against the float64 references (tests/search_ref.py, tests/refine_ref.py)
at the precision fp32 reaches, some 100 times tighter than parity.RTOL.  Each case asserts, through acq_plan_launch,
that it runs the kernel it is named after; where the kernel follows from the total tile count, the whole search runs and
a subset of rows is compared.  test_refine_edges refines records placed where no search puts them."""
import ctypes as C

import numpy as np
import pytest

import flydog_sdr_gps_b200 as F
from flydog_sdr_gps_b200 import _lib, scenarios, synth
from flydog_sdr_gps_b200 import sats as S

from profile_ref import LAGS_E1B, LAGS_L1, circular_distance, peak2_of
from refine_ref import RefineRef, check_fine
from search_ref import NOISE_RTOL, PEAK_RTOL, PROFILE_TAU, Worst, check_cells, check_profile, check_record

pytestmark = pytest.mark.gpu

EXCL = 4
BIN = F.BIN_HZ
# acq_plan_launch's kernel codes
L1, E1B_ONE_CTA, E1B_CLUSTER, L1_MULTI, L1_CR = 0, 1, 2, 3, 6   # E1B_ONE_CTA: k_search_e1b_multi when K > 1


def _case(name):
    """(table, params keywords, captures [n_cap, bytes], sel (None: the table), compared rows [(capture, slot)],
    [(family e1b, kernel, claims or None)])."""
    nav = S.navstar()
    every = [(0, s) for s in range(32)]
    if name == "l1_cr_static_one_capture":   # cfg1: one 1-bit block, the shape whose capture rides in the front end's launch
        return (nav, {}, [synth.make_capture(41, 1, nav, scenarios.signals("cfg1", 3))], None, every, [(0, L1_CR, 0)])
    if name == "l1_cr_chunks_claimed":        # two cfg1 captures: 2624 tiles
        caps = [synth.make_capture(41 + c, 1, nav, scenarios.signals("cfg1", 3 + c)) for c in range(2)]
        return nav, {}, caps, None, [(c, s) for c in range(2) for s in range(c, 32, 3)], [(0, L1_CR, 1)]
    if name in ("l1_half_bins_1bit", "l1_half_bins_2bit"):
        bits = 2 if name.endswith("2bit") else 1
        cap = synth.make_capture(45, 1, nav, scenarios.signals("cfg1", 5), sample_bits=bits)
        return (nav, dict(half_bin=1, dop_lo=-41, dop_hi=40, sample_bits=bits), [cap], None, every[::2] + [(0, 31)],
                [(0, L1, None)])
    if name == "l1_multi_cfg2_four_rows":
        sig = scenarios.signals("cfg2", 2)
        sel = [s[0] for s in sig[:3]] + [31]
        kw = scenarios.params_kw("cfg2")
        return (nav, kw, [synth.make_capture(42, 20, nav, sig)], sel, [(0, s) for s in range(4)], [(0, L1_MULTI, None)])
    if name == "l1_multi_k3_circular":
        sig = [(30, 700, -8.0 * BIN, 45, 0.3), (2, 5000, 11.4 * BIN, 44, 1.0)]
        return (nav, dict(k_noncoh=3, wrap_mode=F.WRAP_CIRCULAR), [synth.make_capture(46, 3, nav, sig)], [2, 30, 31, 7],
                [(0, s) for s in range(4)], [(0, L1_MULTI, None)])
    if name == "l1_multi_k5_half_bins_code_doppler":   # s(4, h) = round(4 h / 770) is -1 from h = -97 down
        sig = [(4, 9000, -55.2 * BIN, 44, 0.2), (11, 300, -60.1 * BIN, 44, 1.0)]
        kw = dict(k_noncoh=5, half_bin=1, dop_lo=-130, dop_hi=-90, code_doppler=1)
        return (nav, kw, [synth.make_capture(44, 5, nav, sig, code_doppler=True)], [4, 11, 19, 31],
                [(0, s) for s in range(4)], [(0, L1_MULTI, None)])
    gal = scenarios.table("cfg3")
    if name in ("e1b_one_cta", "e1b_multi"):
        cfg = "cfg3" if name == "e1b_one_cta" else "cfg3_k4"
        kw = scenarios.params_kw(cfg)
        sig = scenarios.signals(cfg, 2)
        rows = sorted({s[0] for s in sig[:6 if cfg == "cfg3" else 4]} | {0, 49})
        cap = synth.make_capture(47, kw.get("k_noncoh", 1), gal, sig)
        return gal, kw, [cap], None, [(0, s) for s in rows], [(1, E1B_ONE_CTA, 1)]
    if name in ("e1b_cluster_k1", "e1b_cluster_k4"):   # 3 rows x 9 bins: a cluster per tile
        K = 1 if name.endswith("k1") else 4
        sig = [(3, 30001, -2.0 * BIN, 44, 0.1), (20, 12345, 3.3 * BIN, 42, 1.3)]
        return (gal, dict(k_noncoh=K, dop_lo=-4, dop_hi=4), [synth.make_capture(48, K, gal, sig)], [3, 20, 49],
                [(0, s) for s in range(3)], [(1, E1B_CLUSTER, None)])
    if name == "e1b_cluster_k6_code_doppler":   # s(5, h) = round(5 h / 385) is -1 from h = -39 down
        sig = [(3, 30001, -40.2 * BIN, 44, 0.1)]
        kw = dict(k_noncoh=6, dop_lo=-44, dop_hi=-36, code_doppler=1)
        return (gal, kw, [synth.make_capture(49, 6, gal, sig, code_doppler=True)], [3, 20, 49],
                [(0, s) for s in range(3)], [(1, E1B_CLUSTER, None)])
    if name == "mixed_c_a_and_e1b":   # cfg4: the C/A launch, then the E1B launch chained to it
        t4 = scenarios.table("cfg4")
        sig = scenarios.signals("cfg4", 3)
        sel = sorted({s[0] for s in sig} | {0, 31, 32, 81})
        cap = synth.make_capture(41, 1, t4, sig)
        return t4, {}, [cap], sel, [(0, s) for s in range(len(sel))], [(0, L1_CR, 0), (1, E1B_ONE_CTA, None)]
    raise KeyError(name)


CASES = ["l1_cr_static_one_capture", "l1_cr_chunks_claimed", "l1_half_bins_1bit", "l1_half_bins_2bit",
         "l1_multi_cfg2_four_rows", "l1_multi_k3_circular", "l1_multi_k5_half_bins_code_doppler", "e1b_one_cta",
         "e1b_multi", "e1b_cluster_k1", "e1b_cluster_k4", "e1b_cluster_k6_code_doppler", "mixed_c_a_and_e1b"]


def _assert_kernels(eng, table, n_cap, sel, kernels):
    p = eng.params
    rows = range(len(table)) if sel is None else sel
    sms = eng.device_info()["sm_count"]
    plan = _lib.AcqLaunchPlan()
    for e1b, kernel, claims in kernels:
        n_rows = sum((table[s][3] == S.E1B) == bool(e1b) for s in rows)
        assert _lib.load().acq_plan_launch(p.k_noncoh, p.half_bin, e1b, n_cap * n_rows * eng.n_dop, sms, C.byref(plan)) == 0
        assert plan.kernel == kernel and (claims is None or plan.claims == claims), (e1b, plan.kernel, plan.claims)


def check_peak2(pk, P, lag, what):
    """An acq_peak2 row against the reduction of the reference's P: peak2 at PEAK_RTOL, lag2 the reference's or a lag
    outside the lobe whose P is within PEAK_RTOL of its peak2, ratio at PEAK_RTOL + PROFILE_TAU, noise_ex at NOISE_RTOL."""
    peak2, lag2, ratio, noise_ex = peak2_of(P, lag, EXCL)
    assert abs(pk["peak2"] / peak2 - 1) <= PEAK_RTOL, (what, pk["peak2"], peak2)
    g2 = int(pk["lag2"])
    assert g2 == lag2 or (circular_distance(P.size, lag)[g2] > EXCL and P[g2] >= peak2 * (1 - PEAK_RTOL)), (what, g2, lag2)
    assert abs(pk["ratio"] / ratio - 1) <= PEAK_RTOL + PROFILE_TAU, (what, pk["ratio"], ratio)
    assert abs(pk["noise_ex"] / noise_ex - 1) <= NOISE_RTOL, (what, pk["noise_ex"], noise_ex)


@pytest.mark.parametrize("name", CASES)
def test_search_and_profile_at_fp32_precision(gpu_required, oracle, name):
    table, kw, caps, sel, compared, kernels = _case(name)
    with F.AcqEngine(table, F.default_params(**kw)) as eng:
        _assert_kernels(eng, table, len(caps), sel, kernels)
        n0 = eng.launch_count
        rec, grid = eng.search(np.concatenate(caps), sel=None if sel is None else np.array(sel, np.int32), want_grid=True)
        if name == "l1_cr_static_one_capture":   # front end (capture as its argument), forward FFT, search, k_pick_small
            assert eng.launch_count - n0 == 4
        pk, prof = eng.profile(rec, excl=EXCL, want_profile=True)
        off = eng.profile_offsets(len(caps), sel)
        fine = eng.refine(rec)
    oprm = oracle.default_params(**kw)
    refs = [RefineRef(oracle, oprm, cap, table) for cap in caps]
    n_sel = rec.shape[1]
    worst = Worst(name)
    for c, s in compared:
        sat = s if sel is None else sel[s]
        what = "%s capture %d sat %d" % (name, c, sat)
        ref = refs[c].cells(sat)
        check_cells(grid[c, s], ref, worst, what)
        r = rec[c, s]
        check_record(r, ref, worst, what)
        P = ref[5][int(r["dop"]) - int(ref[0][0])]
        i = c * n_sel + s
        check_profile(prof[off[i]:off[i + 1]], P, worst, what)
        check_peak2(pk[c, s], P, int(r["lag"]), what)
        check_fine(fine[c, s], r, refs[c], worst, what)
    print(worst)


# test_refine_edges: three captures of a K = 2, half-bin engine over -9..8 half-bins on the reference table.  Rows: a C/A
# row with a signal (3), a C/A row without one (20), an E1B row with a signal (44) and the last row of the table (E1B
# 58, whose negative bins read the zero row after the table in the reference wrap).
EDGE_SEL = np.array([3, 20, 44, 58], np.int32)
EDGE_KW = dict(k_noncoh=2, half_bin=1, dop_lo=-9, dop_hi=8)


def _edge_records(rec, n_sel, j):
    """Placement j of the records: the search's records with (dop, lag) set per slot to the j-th pair of the cross
    product of dop_lo, dop_lo + 1, dop_hi - 1, dop_hi, the record's dop with lag 0, 1, L - 2, L - 1 and the record's lag
    (slot s starts s pairs further on, so every capture and slot meets every pair)."""
    out = rec.copy()
    lo, hi = EDGE_KW["dop_lo"], EDGE_KW["dop_hi"]
    for c in range(out.shape[0]):
        for s in range(n_sel):
            r = out[c, s]
            L = LAGS_E1B if S.reference_table()[int(r["sat"])][3] == S.E1B else LAGS_L1
            dops = [lo, lo + 1, hi - 1, hi, int(rec[c, s]["dop"])]
            lags = [0, 1, L - 2, L - 1, int(rec[c, s]["lag"])]
            k = (j + s + 7 * c) % 25
            r["dop"], r["lag"] = dops[k // 5], lags[k % 5]
    return out


def test_refine_edges(gpu_required, oracle):
    """acq_refine accepts any record that passes its checks: records at dop_lo and dop_hi and the odd and even half-bin
    indices next to them (d +- 1 one bin past the range), lag 0 (lag n - 1 wraps to N - 1), lags L - 2 and L - 1 of C/A
    and E1B rows, a row without a signal (den small, delta ill-conditioned or clamped), the last table row in the
    reference wrap, and rows of the second and third captures -- every one against RefineRef, peak against the
    reference's sum of |r|^2 at that cell.  acq_refine_device of the same records gives the same bytes."""
    import torch
    table = S.reference_table()
    sig = [[(3, 4001, 3.3 * BIN, 48, 1.0), (44, 30003, -4.2 * BIN, 49, 0.4)],
           [(3, 16000, -4.4 * BIN, 47, 2.0), (44, 100, 3.9 * BIN, 48, 1.1)],
           [(3, 0, 0.6 * BIN, 46, 0.3), (44, 65000, -0.2 * BIN, 48, 2.5)]]
    caps = [synth.make_capture(1300 + c, 2, table, sig[c]) for c in range(3)]
    oprm = oracle.default_params(**EDGE_KW)
    refs = [RefineRef(oracle, oprm, cap, table) for cap in caps]
    worst = Worst("refine edges")
    with F.AcqEngine(table, F.default_params(**EDGE_KW)) as eng:
        rec = eng.search(np.concatenate(caps), sel=EDGE_SEL)
        for j in range(25):
            placed = _edge_records(rec, len(EDGE_SEL), j)
            fine = eng.refine(placed)
            assert (fine["ca_shift"] >= 0).all(), fine
            d_rec = torch.from_numpy(placed.reshape(-1).view(np.uint8).copy()).cuda()
            d_out = torch.zeros(fine.nbytes, dtype=torch.uint8, device="cuda")
            torch.cuda.synchronize()
            eng.refine_device(d_rec.data_ptr(), d_out.data_ptr(), placed.size)
            torch.cuda.synchronize()
            assert d_out.cpu().numpy().tobytes() == fine.tobytes(), j
            for c in range(len(caps)):
                check_fine(fine[c], placed[c], refs[c], worst, "placement %d capture %d" % (j, c))
    print(worst)
