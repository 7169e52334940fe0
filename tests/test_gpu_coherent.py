"""GPU suite (-m gpu) of the coherent search (acq_search_coherent): M = 1 against acq_search_grid bit for bit, M > 1
against the float64 reference (tests/coherent_ref.py), the phase alignment pinned by in-phase signals, data-bit edges,
sensitivity against M = 1 on the same bytes, host and device forms, refusals, and the engine's lifetime."""
import numpy as np
import pytest

import flydog_sdr_gps_b200 as F
from flydog_sdr_gps_b200 import synth
from flydog_sdr_gps_b200 import sats as S

from coherent_ref import CoherentRef, grid_h
from search_ref import Worst, check_cells, check_record

pytestmark = pytest.mark.gpu
BIN = F.BIN_HZ


def _dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a).reshape(-1).view(np.uint8).copy()).cuda()


# (table, params keywords, K, sample_bits, sel) of the M = 1 shapes
def _m1_shape(name):
    nav = S.navstar()
    sbas = nav + [(120, 145, 0, S.SBAS)]
    return {
        "full_bins_k1": (S.reference_table()[:36], {}, 1, 1, None),
        "half_bins_k4": (nav, dict(k_noncoh=4, half_bin=1, dop_lo=-30, dop_hi=27), 4, 1, None),
        "circular_wrap_k4": (nav, dict(k_noncoh=4, wrap_mode=1), 4, 1, np.array([0, 31, 7, 3], np.int32)),
        "two_bit_k1_half_bins": (nav, dict(sample_bits=2, half_bin=1), 1, 2, np.array([7, 3, 12], np.int32)),
        "sbas_row_k2": (sbas, dict(k_noncoh=2), 2, 1, np.array([32, 7, 0], np.int32)),
    }[name]


@pytest.mark.parametrize("name", ["full_bins_k1", "half_bins_k4", "circular_wrap_k4", "two_bit_k1_half_bins", "sbas_row_k2"])
def test_m1_is_acq_search_grid(gpu_required, name):
    """M = 1: records and grid bitwise equal to acq_search_grid on the same engine and bytes (front-end variant path,
    tile decode and accumulation order), over two captures."""
    table, kw, K, bits, sel = _m1_shape(name)
    sig = [(7, 4444, 3.5 * BIN, 45, 0.3), (3, 10000, -11.0 * BIN, 44, 1.7), (0, 8, -19.5 * BIN, 46, 2.5)]
    cap = np.concatenate([synth.make_capture(40 + c, K, table, sig, sample_bits=bits) for c in range(2)])
    with F.AcqEngine(table, F.default_params(**kw)) as eng:
        r0, g0 = eng.search(cap, sel=sel, want_grid=True)
        r1, g1 = eng.search_coherent(cap, 1, sel=sel, want_grid=True)
    assert r1.tobytes() == r0.tobytes()
    assert g1.tobytes() == g0.tobytes()


@pytest.mark.parametrize("m_coh,groups,half_bin", [(m, g, hb) for m in (2, 3, 4, 5) for g in (1, 2) for hb in (0, 1)])
def test_against_reference(gpu_required, oracle, m_coh, groups, half_bin):
    """Cells and records of two satellites (one with a signal, one without) against the float64 reference at
    search_ref's tolerances (check_cells, check_record): peak, noise and snr; the lag wherever the reference's power at
    the search's lag is not within PEAK_RTOL of its peak; the record's dop wherever the reference's runner-up is not
    within SNR_RTOL of its best snr."""
    K = m_coh * groups
    nav = S.navstar()
    kw = dict(k_noncoh=K, half_bin=half_bin, dop_lo=-4 * (1 + half_bin), dop_hi=3 * (1 + half_bin))
    Fv = m_coh * (1 + half_bin)
    h_sig = 2 * Fv + 1
    cap = synth.make_capture(300 + K + half_bin, K, nav, [(9, 3000, h_sig / Fv * BIN, 41, 0.9)])
    sel = np.array([9, 14], np.int32)
    with F.AcqEngine(nav, F.default_params(**kw)) as eng:
        rec, grid = eng.search_coherent(cap, m_coh, sel=sel, want_grid=True)
        p = eng.params
    worst = Worst("coherent M = %d, %d groups, half_bin %d" % (m_coh, groups, half_bin))
    for s, sat in enumerate(sel):
        ref = CoherentRef(oracle, p, cap, nav, int(sat)).cells(m_coh)
        assert np.array_equal(ref[0], grid_h(p, m_coh))
        what = "sat %d" % sat
        check_cells(grid[0, s], ref, worst, what)
        check_record(rec[0, s], ref, worst, what)
    print(worst)
    assert rec[0, 0]["dop"] == h_sig   # the signal row finds its cell


# in-phase points (engine half_bin, M = K, Doppler index h on the coherent grid): integer bins near +-19 and sub-bin v != 0
IN_PHASE = [(0, 5, -95), (0, 5, 95), (0, 5, 97), (0, 5, -93), (0, 4, 4 * 19 + 1), (1, 2, -4 * 19 + 3), (1, 3, 6 * 18 + 5)]


@pytest.mark.parametrize("half_bin,m_coh,h", IN_PHASE)
def test_in_phase_gain(gpu_required, oracle, half_bin, m_coh, h):
    """A strong signal exactly on a coherent grid point: the coherent peak (M = K, G = 1) over the non-coherent peak of
    the same bytes lies in [0.95 M, 1.0 M + eps].  For v = 0 the non-coherent peak is acq_search's record (M = 1 on the
    same engine); for v != 0, where M = 1 has no cell, it is the reference's sum of |r'_b|^2 at the same (d, v).  This pins
    the sign of both terms of theta_j and the sub-bin rotation: the wrong sign of 16 d / N alone gives 0.87 M at h = -95."""
    nav = S.navstar()
    Fv = m_coh * (1 + half_bin)
    cap = synth.make_capture(900 + h, m_coh, nav, [(3, 5000, h / Fv * BIN, 50, 1.1)])
    kw = dict(k_noncoh=m_coh, half_bin=half_bin, dop_lo=-20 * (1 + half_bin), dop_hi=20 * (1 + half_bin))
    with F.AcqEngine(nav, F.default_params(**kw)) as eng:
        rc = eng.search_coherent(cap, m_coh, sel=[3])[0, 0]
        r1 = eng.search(cap, sel=[3])[0, 0]
    assert rc["dop"] == h and rc["lag"] == 1250
    if h % m_coh == 0:
        assert r1["dop"] == h // m_coh and r1["lag"] == 1250
        nc = float(r1["peak"])
    else:
        nc = CoherentRef(oracle, F.default_params(**kw), cap, nav, 3).power(h, m_coh, "noncoh").max()
    ratio = float(rc["peak"]) / nc
    assert 0.95 * m_coh <= ratio <= 1.0 * m_coh + 0.02, ratio


def test_data_bit_edge(gpu_required, oracle):
    """A bit edge at a block boundary inside a group (K = M = 5, edge before block 2): the same record cell as the
    edge-free capture and a peak within 15 % of it; the reference's single-hypothesis sum |T|^2 at that cell collapses
    to a fraction of it."""
    nav = S.navstar()
    h, M = 5 * 7 + 1, 5
    sig = [(3, 5000, h / M * BIN, 47, 0.4)]
    edge = 2 * synth.BLOCK_SAMPLES - synth.BIT_SAMPLES   # bit 0 ends where block 2 begins
    clean = synth.make_capture(17, M, nav, sig)
    flip = synth.make_capture(17, M, nav, sig, data_bits=[1, -1], bit_edge=edge)
    with F.AcqEngine(nav, F.default_params(k_noncoh=M)) as eng:
        rc = eng.search_coherent(clean, M, sel=[3])[0, 0]
        rf = eng.search_coherent(flip, M, sel=[3])[0, 0]
        p = eng.params
    assert (rf["dop"], rf["lag"]) == (rc["dop"], rc["lag"]) == (h, 1250)
    assert 0.85 <= rf["peak"] / rc["peak"] <= 1.15, (rf, rc)
    single = CoherentRef(oracle, p, flip, nav, 3).power(h, M, "single")
    assert single[1250] < 0.2 * rf["peak"], (single[1250], rf["peak"])


# Sensitivity: tools/coherent_bench.py's workload at one C/N0.  A cfg2-shaped engine (K = 20, half-bins, +-80), 128
# captures of 20 blocks with one PRN at a random code phase and Doppler (fixed seeds, so the bytes and the records are
# the same on every run).  Found rates measured once on a B200 (profiles/coherent_bench_b200.json, 29 dB-Hz):
# M = 1 0.523, M = 4 0.625, M = 5 0.680.  "Found" needs no threshold: lag within +-1, Doppler within one coherent step.
SENS_CN0 = 29.0


def _tools():
    import os
    import sys
    tools = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools")
    if tools not in sys.path:
        sys.path.insert(0, tools)
    import coherent_bench
    return coherent_bench


def test_sensitivity(gpu_required):
    import torch
    B = _tools()
    caps, tau, f = B.sensitivity_set(F, S, synth, torch, 1000 + int(SENS_CN0 * 10), 128, SENS_CN0)
    with F.AcqEngine(S.navstar(), F.default_params(**B.CFG2)) as eng:
        rate = {m: float(B.found(F, eng, eng.search_coherent(caps, m, sel=[7])[:, 0], m, tau, f).mean()) for m in (1, 4, 5)}
    print("found rates", rate)
    assert 0.4 <= rate[1] <= 0.65, rate                  # about half the rows at M = 1
    assert rate[4] >= rate[1] + 0.06 and rate[5] >= rate[1] + 0.12, rate


def test_host_and_device_forms(gpu_required):
    """Host and device forms give the same bytes, on the engine stream and on a torch stream; a coherent search between
    two acq_search calls leaves the second bitwise equal to the first."""
    import torch
    nav = S.navstar()
    cap = np.concatenate([synth.make_capture(70 + c, 4, nav, [(5, 800 + 4 * c, (2.25 - c) * BIN, 44, 0.0)]) for c in range(3)])
    sel = np.array([5, 6, 20], np.int32)
    with F.AcqEngine(nav, F.default_params(k_noncoh=4, half_bin=1)) as eng:
        first = eng.search(cap, sel=sel)
        for m in (1, 2, 4):
            host = eng.search_coherent(cap, m, sel=sel)
            d_in = _dev(cap)
            d_out = torch.zeros(host.nbytes, dtype=torch.uint8, device="cuda")
            torch.cuda.synchronize()
            eng.search_coherent_device(d_in.data_ptr(), m, d_out.data_ptr(), 3, sel=sel)
            torch.cuda.synchronize()
            assert d_out.cpu().numpy().tobytes() == host.tobytes()
            st = torch.cuda.Stream()
            d_out.zero_()
            torch.cuda.synchronize()
            eng.search_coherent_device(d_in.data_ptr(), m, d_out.data_ptr(), 3, sel=sel, stream_ptr=st.cuda_stream)
            st.synchronize()
            assert d_out.cpu().numpy().tobytes() == host.tobytes()
            assert eng.search(cap, sel=sel).tobytes() == first.tobytes()
        with F.AcqEngine(nav, F.default_params(k_noncoh=4, half_bin=1)) as fresh:
            assert fresh.search(cap, sel=sel).tobytes() == first.tobytes()


def test_refusals_and_cleared_spectra(gpu_required):
    """E1B rows and code_doppler engines: ACQ_ERR_UNSUPPORTED with nothing launched, the engine still usable;
    k_noncoh % m_coh: ACQ_ERR_ARG; after a coherent search acq_refine*, acq_profile* are ACQ_ERR_ARG until acq_search."""
    import torch
    table = S.reference_table()
    cap = synth.make_capture(5, 4, table, [(2, 4000, 4 * BIN, 48, 1.0)])
    with F.AcqEngine(table, F.default_params(k_noncoh=4)) as eng:
        rec = eng.search(cap, sel=[2, 3])
        n0 = eng.launch_count
        for call in (lambda: eng.search_coherent(cap, 2, sel=[2, 40]), lambda: eng.search_coherent(cap, 2)):
            with pytest.raises(F.AcqError) as ei:
                call()
            assert ei.value.code == -4 and "E1B" in str(ei.value)
        d_in = _dev(cap)
        d_out = torch.zeros(2 * 24, dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()
        with pytest.raises(F.AcqError) as ei:
            eng.search_coherent_device(d_in.data_ptr(), 2, d_out.data_ptr(), 1, sel=[44, 2])
        assert ei.value.code == -4
        with pytest.raises(F.AcqError) as ei:
            eng.search_coherent(cap, 3, sel=[2])
        assert ei.value.code == -1 and "multiple" in str(ei.value)
        assert eng.launch_count == n0
        assert eng.refine(rec).shape == rec.shape   # the refused calls left the last search's spectra alone
        eng.search_coherent(cap, 2, sel=[2, 3])
        d_rec = _dev(rec)
        d_fine = torch.zeros(2 * 16, dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()
        for call in (lambda: eng.refine(rec), lambda: eng.profile(rec),
                     lambda: eng.refine_device(d_rec.data_ptr(), d_fine.data_ptr(), 2),
                     lambda: eng.profile_device(d_rec.data_ptr(), d_fine.data_ptr(), 2)):
            with pytest.raises(F.AcqError) as ei:
                call()
            assert ei.value.code == -1
        assert eng.search(cap, sel=[2, 3]).tobytes() == rec.tobytes()
        assert eng.refine(rec).shape == rec.shape
    nav = S.navstar()
    cap2 = synth.make_capture(6, 4, nav, [(2, 4000, 4 * BIN, 48, 1.0)])
    with F.AcqEngine(nav, F.default_params(k_noncoh=4, code_doppler=1)) as eng:
        r = eng.search(cap2, sel=[2])
        n0 = eng.launch_count
        with pytest.raises(F.AcqError) as ei:
            eng.search_coherent(cap2, 2, sel=[2])
        assert ei.value.code == -4 and "code_doppler" in str(ei.value)
        assert eng.launch_count == n0
        assert eng.search(cap2, sel=[2]).tobytes() == r.tobytes()


def test_engine_lifetime(gpu_required):
    """acq_create / host and device coherent searches / acq_destroy, thirty times: device memory returns to where it was."""
    import torch
    nav = S.navstar()
    cap = synth.make_capture(12, 4, nav, [(2, 4000, 4 * BIN, 48, 1.0)])
    d_in = _dev(cap)
    d_rec = torch.zeros(32 * 24, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()

    def cycle():
        with F.AcqEngine(nav, F.default_params(k_noncoh=4, half_bin=1)) as eng:
            for m in (1, 2, 4):
                r = eng.search_coherent(cap, m)
                eng.search_coherent_device(d_in.data_ptr(), m, d_rec.data_ptr(), 1)
                torch.cuda.synchronize()
                assert d_rec.cpu().numpy().tobytes() == r.tobytes()
    cycle()
    torch.cuda.synchronize()
    free0 = torch.cuda.mem_get_info()[0]
    for _ in range(30):
        cycle()
    torch.cuda.synchronize()
    assert free0 - torch.cuda.mem_get_info()[0] < (32 << 20)
