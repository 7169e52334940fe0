"""GPU suite (-m gpu) of the precision tier: every non-coherent search kernel's cells, records, lag profiles and
second-peak rows against the float64 reference (tests/search_ref.py) at the precision fp32 reaches, some 100 times
tighter than parity.RTOL.  Each case asserts, through acq_plan_launch, that it runs the kernel it is named after; where
the kernel follows from the total tile count, the whole search runs and a subset of rows is compared."""
import ctypes as C

import numpy as np
import pytest

import flydog_sdr_gps_b200 as F
from flydog_sdr_gps_b200 import _lib, scenarios, synth
from flydog_sdr_gps_b200 import sats as S

from profile_ref import circular_distance, peak2_of
from search_ref import (NOISE_RTOL, PEAK_RTOL, PROFILE_TAU, SearchRef, Worst, check_cells, check_profile,
                        check_record)

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
    oprm = oracle.default_params(**kw)
    refs = [SearchRef(oracle, oprm, cap, table) for cap in caps]
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
    print(worst)
