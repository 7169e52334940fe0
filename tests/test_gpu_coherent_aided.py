"""GPU suite (-m gpu) of the aided coherent search (acq_search_coherent_aided / acq_search_coherent_aided_device): every
(capture, satellite) row searched coherently over its own window of the coherent Doppler grid.  The window cells are the
full coherent search's cells to the byte, the records are Correlate()'s rule over the window, M = 1 is acq_search_aided,
and the cells agree with the float64 reference (tests/coherent_ref.py)."""
import numpy as np
import pytest

import flydog_sdr_gps_b200 as F
from flydog_sdr_gps_b200 import _lib, synth
from flydog_sdr_gps_b200 import sats as S

from coherent_ref import CoherentRef
from search_ref import Worst
from test_gpu_coherent_sweep import check_cells, check_record

pytestmark = pytest.mark.gpu
BIN = F.BIN_HZ
INT32_MIN, INT32_MAX = -2 ** 31, 2 ** 31 - 1
SBAS_ROW = 32


def window_lo(center, hw, dop_lo, dop_hi):
    return int(min(max(int(center) - hw, dop_lo), dop_hi - 2 * hw))


def window_pick(cells, lo, sat):
    """Correlate()'s rule over one row's window: largest snr > 0, first (lowest Doppler) on ties; else zeros."""
    r = np.zeros(1, F.RECORD_DTYPE)[0]
    r["sat"] = sat
    best, bd = 0.0, -1
    for j in range(len(cells)):
        if cells["snr"][j] > best:
            best, bd = cells["snr"][j], j
    if bd >= 0:
        c = cells[bd]
        r["lag"], r["dop"], r["peak"], r["noise"], r["snr"] = c["lag"], lo + bd, c["peak"], c["noise"], c["snr"]
    return r


def coh_range(p, m):
    return m * p.dop_lo, m * p.dop_hi


def check_against_full(p, m, rec, grid, full_grid, centers, hw, sel):
    """Every aided cell j of row r is the full coherent grid's cell at lo_r + j, byte for byte, and every record is the
    window pick of its own cells."""
    clo, chi = coh_range(p, m)
    n_cap, n_sel, W = grid.shape
    assert W == 2 * hw + 1 and rec.shape == (n_cap, n_sel) and full_grid.shape[2] == chi - clo + 1
    for c in range(n_cap):
        for s in range(n_sel):
            lo = window_lo(centers[c, s], hw, clo, chi)
            assert clo <= lo and lo + W - 1 <= chi
            assert grid[c, s].tobytes() == full_grid[c, s, lo - clo: lo - clo + W].tobytes(), (c, s, lo)
            assert rec[c, s].tobytes() == window_pick(grid[c, s], lo, sel[s]).tobytes(), (c, s, lo)


def _table():
    """32 Navstar rows, an SBAS row (no replica: a zero code row) and the 4 QZSS rows."""
    return S.navstar() + [(120, 145, 0o1106, S.SBAS)] + S.qzss()


def _dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a).reshape(-1).view(np.uint8).copy()).cuda()


# ---------------------------------------------------------------- seeded sweep
RANGE_KINDS = ["symmetric", "asymmetric", "positive", "negative", "single"]


def _case(seed):
    rng = np.random.default_rng(8300 + seed)
    M, G = 1 + seed % 5, int(rng.integers(1, 4))
    half = int(rng.integers(0, 2))
    bits = int(rng.choice([1, 2]))
    wrap = int(rng.integers(0, 2))
    kind = RANGE_KINDS[seed % 5]
    if kind == "symmetric":
        hi = int(rng.integers(1, 4)) * (1 + half)
        lo = -hi
    elif kind == "asymmetric":
        lo = -1 - int(rng.integers(0, 3))
        hi = -lo + 1 + int(rng.integers(0, 3))
    elif kind == "positive":
        lo = int(rng.integers(0, 20))
        hi = lo + int(rng.integers(1, 4))
    elif kind == "negative":
        hi = -int(rng.integers(0, 20))
        lo = hi - int(rng.integers(1, 4))
    else:
        lo = hi = int(rng.integers(-15, 16))
    table = _table()
    sel = [int(s) for s in rng.choice(len(table), int(rng.integers(1, 5)), replace=False)]
    if seed % 3 == 1 and SBAS_ROW not in sel:
        sel[0] = SBAS_ROW
    n_cap = int(rng.integers(1, 4))
    step = BIN / (1 + half)
    present = [s for s in sel if s != SBAS_ROW] or [0]
    caps = []
    for c in range(n_cap):
        sig = [(int(s), int(rng.integers(0, 16368)), float(rng.uniform(lo - 0.3, hi + 0.3)) * step,
                float(rng.uniform(43, 48)), float(rng.uniform(0, 2 * np.pi)))
               for s in rng.choice(present, min(len(present), 1 + c % 2), replace=False)]
        caps.append(synth.make_capture(8400 + 10 * seed + c, M * G, table, sig, sample_bits=bits))
    kw = dict(k_noncoh=M * G, half_bin=half, sample_bits=bits, wrap_mode=wrap, dop_lo=lo, dop_hi=hi)
    n_dop_c = M * (hi - lo) + 1
    # half_width from 0 up to (n_dop_c - 1) / 2: both ends on some seeds, random on the others
    hw = [0, (n_dop_c - 1) // 2][seed % 2] if seed < 4 else int(rng.integers(0, (n_dop_c - 1) // 2 + 1))
    clo, chi = M * lo, M * hi
    choices = [clo, chi, clo - 3, chi + 3, clo - 1000, chi + 1000, INT32_MIN, INT32_MAX]
    centers = np.array([[int(rng.integers(clo, chi + 1)) if rng.random() < 0.5 else int(rng.choice(choices))
                         for _ in sel] for _ in range(n_cap)], np.int32)
    centers.reshape(-1)[:2] = [INT32_MIN, INT32_MAX][:centers.size]
    return table, kw, M, np.array(sel, np.int32), caps, centers, hw


@pytest.mark.parametrize("seed", range(10))
def test_window_cells_are_the_full_coherent_cells(gpu_required, seed):
    """M = 1..5, 1-3 groups, half-bins, 2-bit captures, both wraps, SBAS rows, 1-3 captures, symmetric, asymmetric,
    one-sided and single-bin ranges; centres inside, at both ends, beyond them and at INT32_MIN / INT32_MAX."""
    table, kw, M, sel, caps, centers, hw = _case(seed)
    cap = np.concatenate(caps)
    with F.AcqEngine(table, F.default_params(**kw)) as eng:
        full_r, full_g = eng.search_coherent(cap, M, sel=sel, want_grid=True)
        rec, grid = eng.search_coherent_aided(cap, M, centers, hw, sel=sel, want_grid=True)
        alone = eng.search_coherent_aided(cap, M, centers, hw, sel=sel)   # records alone: the same bytes
        p = eng.params
    check_against_full(p, M, rec, grid, full_g, centers, hw, sel)
    assert alone.tobytes() == rec.tobytes()


def test_whole_range_window_is_the_full_coherent_search(gpu_required):
    """W = n_dop_c on a symmetric range: records and grid bitwise those of acq_search_coherent, whatever the centres."""
    nav = S.navstar()
    sel = np.array([3, 7, 20], np.int32)
    for kw, M in ((dict(k_noncoh=4, dop_lo=-6, dop_hi=6), 4), (dict(k_noncoh=6, half_bin=1, dop_lo=-8, dop_hi=8), 3)):
        K = kw["k_noncoh"]
        cap = np.concatenate([synth.make_capture(60 + c, K, nav, [(7, 3000 + 8 * c, (1.3 - c) * BIN, 44, 0.7)]) for c in range(2)])
        with F.AcqEngine(nav, F.default_params(**kw)) as eng:
            full_r, full_g = eng.search_coherent(cap, M, sel=sel, want_grid=True)
            hw = (eng.coherent_dops(M) - 1) // 2
            rng = np.random.default_rng(M)
            for centers in (np.zeros((2, 3), np.int32), rng.integers(-1000, 1000, (2, 3)).astype(np.int32)):
                rec, grid = eng.search_coherent_aided(cap, M, centers, hw, sel=sel, want_grid=True)
                assert rec.tobytes() == full_r.tobytes() and grid.tobytes() == full_g.tobytes()


@pytest.mark.parametrize("kw", [dict(), dict(k_noncoh=4, half_bin=1, dop_lo=-30, dop_hi=27)], ids=["k1_full_bins", "k4_half_bins"])
def test_m1_is_acq_search_aided(gpu_required, kw):
    """M = 1 gives acq_search_aided's records and grid on the same engine, bytes, centres and half_width: with K = 1 on
    full bins the aided search runs on k_search_l1_cr, with K = 4 on half-bins on k_search_l1_multi."""
    nav = S.navstar()
    K = kw.get("k_noncoh", 1)
    caps = np.concatenate([synth.make_capture(90 + c, K, nav, [(4, 1000 + 40 * c, (5.5 - 3 * c) * BIN, 46, 1.0),
                                                                 (11, 9000, -12.0 * BIN, 45, 0.2)]) for c in range(3)])
    rng = np.random.default_rng(11)
    with F.AcqEngine(nav, F.default_params(**kw)) as eng:
        p = eng.params
        centers = rng.integers(p.dop_lo - 5, p.dop_hi + 6, (3, 32)).astype(np.int32)
        for hw in (0, 2, 5):
            want_r, want_g = eng.search_aided(caps, centers, hw, want_grid=True)
            rec, grid = eng.search_coherent_aided(caps, 1, centers, hw, want_grid=True)
            assert rec.tobytes() == want_r.tobytes() and grid.tobytes() == want_g.tobytes(), hw


@pytest.mark.parametrize("m_coh,groups,half_bin", [(2, 2, 0), (3, 1, 1), (4, 2, 1), (5, 1, 0)])
def test_windows_against_reference(gpu_required, oracle, m_coh, groups, half_bin):
    """Windowed rows (a signal row and a noise row, one window at the range's edge) against the float64 reference with
    search_ref's tolerances (test_gpu_coherent_sweep.check_cells); each record against the reference's window pick."""
    K = m_coh * groups
    nav = S.navstar()
    kw = dict(k_noncoh=K, half_bin=half_bin, dop_lo=-4 * (1 + half_bin), dop_hi=3 * (1 + half_bin))
    Fv = m_coh * (1 + half_bin)
    h_sig = 2 * Fv + 1
    cap = synth.make_capture(500 + K + half_bin, K, nav, [(9, 3000, h_sig / Fv * BIN, 41, 0.9)])
    sel = np.array([9, 14], np.int32)
    hw = m_coh
    centers = np.array([[h_sig + 1, INT32_MIN]], np.int32)
    with F.AcqEngine(nav, F.default_params(**kw)) as eng:
        rec, grid = eng.search_coherent_aided(cap, m_coh, centers, hw, sel=sel, want_grid=True)
        p = eng.params
    clo, chi = coh_range(p, m_coh)
    base = CoherentRef(oracle, p, cap, nav, 9)
    worst = Worst("aided coherent M = %d, %d groups, half_bin %d" % (m_coh, groups, half_bin))
    for s, sat in enumerate(sel):
        lo = window_lo(centers[0, s], hw, clo, chi)
        hs_w = np.arange(lo, lo + 2 * hw + 1)
        hs, snr = check_cells(grid[0, s], base.for_sat(int(sat)), m_coh, hs=hs_w, worst=worst, what="sat %d" % sat)
        check_record(rec[0, s], grid[0, s], hs, snr)
    print(worst)
    assert rec[0, 0]["dop"] == h_sig   # the signal row finds its cell inside its window


def _tools():
    import os
    import sys
    tools = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools")
    if tools not in sys.path:
        sys.path.insert(0, tools)
    import coherent_bench
    return coherent_bench


def truth_centers(eng, m_coh, f_hz, seed):
    """Centres on the coherent grid: the true Doppler's index plus a seeded offset of at most M steps (one engine
    half-bin).  With half_width = 2 M every window holds the truth +- M steps."""
    Fv = m_coh * (1 + eng.params.half_bin)
    h = np.round(np.asarray(f_hz) * Fv / BIN).astype(np.int64)
    off = np.random.default_rng(seed).integers(-m_coh, m_coh + 1, h.size)
    return (h + off).astype(np.int32)


def test_same_records_on_the_sensitivity_workload(gpu_required):
    """coherent_bench's sensitivity set (cfg2 shape, 128 captures, 29 dB-Hz, M = 5): wherever the full coherent search's
    record lies inside the row's window the aided record is the same bytes, and every row the full search finds the
    aided search finds too."""
    import torch
    B = _tools()
    M = 5
    caps, tau, f = B.sensitivity_set(F, S, synth, torch, 1000 + 290, 128, 29.0)
    with F.AcqEngine(S.navstar(), F.default_params(**B.CFG2)) as eng:
        full = eng.search_coherent(caps, M, sel=[7])[:, 0]
        centers = truth_centers(eng, M, f, 29)
        hw = 2 * M
        aided = eng.search_coherent_aided(caps, M, centers.reshape(-1, 1), hw, sel=[7])[:, 0]
        clo, chi = coh_range(eng.params, M)
        found_full = B.found(F, eng, full, M, tau, f)
        found_aided = B.found(F, eng, aided, M, tau, f)
    inside = 0
    for i in range(128):
        lo = window_lo(centers[i], hw, clo, chi)
        if lo <= full[i]["dop"] <= lo + 2 * hw:
            inside += 1
            assert aided[i].tobytes() == full[i].tobytes(), i
        if found_full[i]:
            assert found_aided[i], i
    print("found rates: full %.3f aided %.3f (%d of 128 full records inside the window)"
          % (found_full.mean(), found_aided.mean(), inside))
    assert found_aided.mean() >= found_full.mean()


def test_launch_policies(gpu_required):
    """One search of a single wave (static stride: no more tiles than SMs) and one long enough to claim tiles from the
    counter (at least 6 tiles per CTA): both give the full coherent search's cells in every window."""
    nav = S.navstar()
    kw = dict(k_noncoh=2, half_bin=1, dop_lo=-10, dop_hi=10)
    M = 2
    caps = np.concatenate([synth.make_capture(700 + c, 2, nav, [(c % 32, 4 * (100 + 37 * c), (3.5 - c) * BIN, 45, 0.1 * c)])
                           for c in range(8)])
    rng = np.random.default_rng(21)
    with F.AcqEngine(nav, F.default_params(**kw)) as eng:
        sms = eng.device_info()["sm_count"]
        p = eng.params
        clo, chi = coh_range(p, M)
        # single wave: 1 capture x 4 satellites x W = 5
        sel = np.array([0, 1, 2, 3], np.int32)
        one = caps[:2 * 8192]
        full_r, full_g = eng.search_coherent(one, M, sel=sel, want_grid=True)
        centers = rng.integers(clo - 3, chi + 4, (1, 4)).astype(np.int32)
        rec, grid = eng.search_coherent_aided(one, M, centers, 2, sel=sel, want_grid=True)
        assert 4 * 5 <= sms
        check_against_full(p, M, rec, grid, full_g, centers, 2, sel)
        # claimed: 8 captures x 32 satellites x W = 9
        full_r, full_g = eng.search_coherent(caps, M, want_grid=True)
        centers = rng.integers(clo - 3, chi + 4, (8, 32)).astype(np.int32)
        rec, grid = eng.search_coherent_aided(caps, M, centers, 4, want_grid=True)
        assert 8 * 32 * 9 >= 6 * sms
        check_against_full(p, M, rec, grid, full_g, centers, 4, np.arange(32))
        for _ in range(2):   # the tile counters come back to zero after each claiming launch
            assert eng.search_coherent_aided(caps, M, centers, 4).tobytes() == rec.tobytes()


def test_host_and_device_forms(gpu_required):
    """Host and device forms give the same bytes, on the engine stream and on a torch stream; a coherent aided search
    between two acq_search calls leaves the second bitwise equal to the first."""
    import torch
    nav = S.navstar()
    cap = np.concatenate([synth.make_capture(70 + c, 4, nav, [(5, 800 + 4 * c, (2.25 - c) * BIN, 44, 0.0)]) for c in range(3)])
    sel = np.array([5, 6, 20], np.int32)
    rng = np.random.default_rng(31)
    with F.AcqEngine(nav, F.default_params(k_noncoh=4, half_bin=1)) as eng:
        first = eng.search(cap, sel=sel)
        for m in (1, 2, 4):
            centers = rng.integers(-45 * m, 45 * m, (3, 3)).astype(np.int32)
            host = eng.search_coherent_aided(cap, m, centers, 2 * m, sel=sel)
            d_in = _dev(cap)
            d_c = _dev(centers)
            d_out = torch.zeros(host.nbytes, dtype=torch.uint8, device="cuda")
            torch.cuda.synchronize()
            eng.search_coherent_aided_device(d_in.data_ptr(), m, d_c.data_ptr(), 2 * m, d_out.data_ptr(), 3, sel=sel)
            torch.cuda.synchronize()
            assert d_out.cpu().numpy().tobytes() == host.tobytes()
            st = torch.cuda.Stream()
            d_out.zero_()
            torch.cuda.synchronize()
            eng.search_coherent_aided_device(d_in.data_ptr(), m, d_c.data_ptr(), 2 * m, d_out.data_ptr(), 3, sel=sel,
                                             stream_ptr=st.cuda_stream)
            st.synchronize()
            assert d_out.cpu().numpy().tobytes() == host.tobytes()
            assert eng.search(cap, sel=sel).tobytes() == first.tobytes()


def test_refusals_and_cleared_spectra(gpu_required):
    """E1B rows and code_doppler engines: ACQ_ERR_UNSUPPORTED; W > n_dop_c, half_width < 0, NULL centres and
    k_noncoh % m_coh: ACQ_ERR_ARG.  Nothing is launched and the engine stays usable.  After an aided coherent search
    acq_refine*, acq_profile* are ACQ_ERR_ARG until acq_search."""
    import torch
    L = _lib.load()
    table = S.reference_table()
    cap = synth.make_capture(5, 4, table, [(2, 4000, 4 * BIN, 48, 1.0)])
    c2 = np.zeros((1, 2), np.int32)
    with F.AcqEngine(table, F.default_params(k_noncoh=4)) as eng:
        rec = eng.search(cap, sel=[2, 3])
        n0 = eng.launch_count
        n_dop_c = eng.coherent_dops(2)
        with pytest.raises(F.AcqError) as ei:
            eng.search_coherent_aided(cap, 2, c2, 1, sel=[2, 40])
        assert ei.value.code == -4 and "E1B" in str(ei.value)
        d_in = _dev(cap)
        d_c = _dev(c2)
        d_out = torch.zeros(2 * 24, dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()
        with pytest.raises(F.AcqError) as ei:
            eng.search_coherent_aided_device(d_in.data_ptr(), 2, d_c.data_ptr(), 1, d_out.data_ptr(), 1, sel=[44, 2])
        assert ei.value.code == -4
        for hw, text in (((n_dop_c + 1) // 2, "exceeds n_dop_c"), (-1, "half_width must be >= 0")):
            with pytest.raises(F.AcqError) as ei:
                eng.search_coherent_aided(cap, 2, c2, hw, sel=[2, 3])
            assert ei.value.code == -1 and text in str(ei.value)
        assert eng.launch_count == n0
        assert eng.refine(rec).shape == rec.shape
        eng.search_coherent_aided(cap, 2, c2, (n_dop_c - 1) // 2, sel=[2, 3])   # W = n_dop_c is accepted
        eng.search(cap, sel=[2, 3])
        n0 = eng.launch_count
        out = np.zeros(2, F.RECORD_DTYPE)
        sel = np.array([2, 3], np.int32)
        assert L.acq_search_coherent_aided(eng._h, cap.ctypes.data, 1, sel.ctypes.data, 2, 2, None, 1, out.ctypes.data,
                                           None) == -1
        assert b"dop_center is NULL" in L.acq_last_error()
        with pytest.raises(F.AcqError) as ei:
            eng.search_coherent_aided(cap, 3, c2, 1, sel=[2, 3])
        assert ei.value.code == -1 and "multiple" in str(ei.value)
        assert eng.launch_count == n0
        assert eng.refine(rec).shape == rec.shape   # the refused calls left the last search's spectra alone
        eng.search_coherent_aided(cap, 2, c2, 1, sel=[2, 3])
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
            eng.search_coherent_aided(cap2, 2, np.zeros(1, np.int32), 1, sel=[2])
        assert ei.value.code == -4 and "code_doppler" in str(ei.value)
        assert eng.launch_count == n0
        assert eng.search(cap2, sel=[2]).tobytes() == r.tobytes()


def test_engine_lifetime(gpu_required):
    """acq_create / host and device aided coherent searches / acq_destroy, thirty times: device memory returns to where
    it was."""
    import torch
    nav = S.navstar()
    cap = synth.make_capture(12, 4, nav, [(2, 4000, 4 * BIN, 48, 1.0)])
    centers = np.arange(-48, 48, 3, dtype=np.int32)
    d_in = _dev(cap)
    d_c = _dev(centers)
    d_rec = torch.zeros(32 * 24, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()

    def cycle():
        with F.AcqEngine(nav, F.default_params(k_noncoh=4, half_bin=1)) as eng:
            for m in (1, 2, 4):
                r = eng.search_coherent_aided(cap, m, centers, m)
                eng.search_coherent_aided_device(d_in.data_ptr(), m, d_c.data_ptr(), m, d_rec.data_ptr(), 1)
                torch.cuda.synchronize()
                assert d_rec.cpu().numpy().tobytes() == r.tobytes()
    cycle()
    torch.cuda.synchronize()
    free0 = torch.cuda.mem_get_info()[0]
    for _ in range(30):
        cycle()
    torch.cuda.synchronize()
    assert free0 - torch.cuda.mem_get_info()[0] < (32 << 20)


def test_capture_farm_coherent(gpu_required):
    """A one-rank CaptureFarm with m_coh returns search_coherent's bytes, and with half_width as well
    search_coherent_aided's."""
    import torch
    from flydog_sdr_gps_b200 import farm
    nav = S.navstar()
    M, K = 2, 4
    caps = np.stack([synth.make_capture(300 + c, K, nav, [(c, 4 * (500 + c), (c - 2.5) * BIN, 45, 0.3)]) for c in range(5)])
    centers = np.random.default_rng(7).integers(-40, 41, (5, 32)).astype(np.int32)
    with F.AcqEngine(nav, F.default_params(k_noncoh=K)) as eng:
        want_full = eng.search_coherent(caps.reshape(-1), M)
        want_aided = eng.search_coherent_aided(caps.reshape(-1), M, centers, 3)
        st = torch.cuda.Stream()
        with torch.cuda.stream(st):
            f = farm.CaptureFarm(eng, 5, K * 8192, 32, m_coh=M)
            f.load(caps)
            full = f.search().copy()
            fa = farm.CaptureFarm(eng, 5, K * 8192, 32, m_coh=M, half_width=3)
            fa.load(caps, dop_center=centers)
            aided = fa.search().copy()
            fa.search_resident()
            st.synchronize()
            res = fa.d_all.cpu().numpy().view(F.RECORD_DTYPE).reshape(5, 32)
    assert full.shape == (5, 32) and aided.shape == (5, 32)
    assert full.tobytes() == want_full.tobytes()
    assert aided.tobytes() == want_aided.tobytes() and res.tobytes() == want_aided.tobytes()
