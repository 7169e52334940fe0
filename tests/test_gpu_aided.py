"""GPU suite (-m gpu) of the aided search: every (capture, satellite) row searched over its own Doppler window
(acq_search_aided / acq_search_aided_device).  The window cells are the full search's cells, the records are
Correlate()'s rule over the window, and every kernel path and library variant agrees."""
import ctypes as C

import numpy as np
import pytest

import flydog_sdr_gps_b200 as F
from flydog_sdr_gps_b200 import _lib, scenarios, synth
from flydog_sdr_gps_b200 import sats as S

from parity import compare_records

pytestmark = pytest.mark.gpu


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


def check_against_full(eng, rec, grid, full_grid, centers, hw, sel, table):
    """Every aided cell is the full grid's cell at lo_r + j (C/A bytewise; E1B peak/lag bytewise, noise/snr 2e-6), and
    every record is the window pick of its own cells."""
    p = eng.params
    sel = np.arange(len(table)) if sel is None else np.asarray(sel)
    n_cap, n_sel, W = grid.shape
    assert W == 2 * hw + 1 and rec.shape == (n_cap, n_sel)
    for c in range(n_cap):
        for s in range(n_sel):
            lo = window_lo(centers[c, s], hw, p.dop_lo, p.dop_hi)
            want = full_grid[c, s, lo - p.dop_lo: lo - p.dop_lo + W]
            got = grid[c, s]
            if table[sel[s]][3] == S.E1B:
                assert np.array_equal(got["peak"], want["peak"]) and np.array_equal(got["lag"], want["lag"]), (c, s)
                for f in ("noise", "snr"):
                    np.testing.assert_allclose(got[f], want[f], rtol=2e-6, equal_nan=True)
            else:
                assert got.tobytes() == want.tobytes(), (c, s, lo)
            assert rec[c, s].tobytes() == window_pick(got, lo, sel[s]).tobytes(), (c, s)


def symmetric_full_window(eng, table, cap, sel=None):
    """W = n_dop on a symmetric range: records and grid bytewise equal to acq_search_grid."""
    p = eng.params
    assert p.dop_lo == -p.dop_hi
    n_sel = len(table) if sel is None else len(sel)
    n_cap = cap.size // (eng.k_noncoh * eng.block_bytes)
    full_r, full_g = eng.search(cap, sel=sel, want_grid=True)
    rng = np.random.default_rng(1)
    for centers in (np.zeros((n_cap, n_sel), np.int32), rng.integers(-1000, 1000, (n_cap, n_sel)).astype(np.int32)):
        rec, grid = eng.search_aided(cap, centers, p.dop_hi, sel=sel, want_grid=True)
        assert rec.tobytes() == full_r.tobytes() and grid.tobytes() == full_g.tobytes()


def test_window_equal_to_range_is_the_full_search(gpu_required):
    nav = S.navstar()
    with F.AcqEngine(nav) as eng:   # cfg1
        symmetric_full_window(eng, nav, synth.make_capture(1, 1, nav, scenarios.signals("cfg1", 1)))
    t4 = scenarios.table("cfg4")   # cfg4: C/A and E1B rows
    with F.AcqEngine(t4) as eng:
        symmetric_full_window(eng, t4, synth.make_capture(41, 1, t4, scenarios.signals("cfg4", 1)))
    kw = dict(scenarios.params_kw("cfg2"), code_doppler=1)   # cfg2's shape: half-bins, K = 20, code-Doppler copies
    with F.AcqEngine(nav, F.default_params(**kw)) as eng:
        cap = synth.make_capture(21, kw["k_noncoh"], nav, scenarios.signals("cfg2", 1), code_doppler=True)
        symmetric_full_window(eng, nav, cap, sel=np.array([0, 5, 9, 17, 30], np.int32))
    t3 = scenarios.table("cfg3_k4")   # cfg3 with K = 4
    kw = scenarios.params_kw("cfg3_k4")
    with F.AcqEngine(t3, F.default_params(**kw)) as eng:
        cap = synth.make_capture(31, kw["k_noncoh"], t3, scenarios.signals("cfg3_k4", 1))
        symmetric_full_window(eng, t3, cap, sel=np.arange(0, 50, 5, dtype=np.int32))


@pytest.mark.parametrize("seed", range(10))
def test_randomized_windows_equal_full_search_and_oracle(gpu_required, oracle, seed):
    """Seeded sweep: Doppler range, half-bins, K, wrap mode, 2-bit captures, code-Doppler, mixed selections, several
    captures with their own centres -- inside, at both edges and outside the range."""
    rng = np.random.default_rng(7100 + seed)
    table = S.reference_table()
    half = int(rng.integers(0, 2))
    K = int(rng.choice([1, 1, 2, 3]))
    span = int(rng.integers(2, 30)) * (2 if half else 1)
    lo = -int(rng.integers(0, span + 1))
    hi = lo + span
    bits = int(rng.choice([1, 2]))
    kw = dict(dop_lo=lo, dop_hi=hi, half_bin=half, k_noncoh=K, wrap_mode=int(rng.integers(0, 2)), sample_bits=bits,
              code_doppler=int(rng.integers(0, 2)), thr_l1=16.0 if K == 1 else 6.0, thr_e1b=16.0 if K == 1 else 6.0)
    sel = rng.choice(len(table), size=int(rng.integers(1, 7)), replace=False).astype(np.int32)
    hw = int(rng.integers(0, span // 2 + 1))
    n_cap = int(rng.integers(1, 4))
    step = F.BIN_HZ / (2 if half else 1)
    caps, sigs = [], []
    for c in range(n_cap):
        sig = []
        for s in sel[:3]:
            period = 65472 if table[s][3] == S.E1B else 16368
            sig.append((int(s), int(rng.integers(0, period)), float(rng.uniform(lo, hi)) * step, float(rng.uniform(44, 50)),
                        float(rng.uniform(0, 6.28))))
        sigs.append(sig)
        caps.append(synth.make_capture(600 + 10 * seed + c, K, table, sig, sample_bits=bits, code_doppler=bool(kw["code_doppler"])))
    choices = [lo, hi, lo - 7, hi + 7, -2 ** 31, 2 ** 31 - 1]   # edges and beyond
    centers = np.array([[int(rng.integers(lo, hi + 1)) if rng.random() < 0.6 else int(rng.choice(choices))
                         for _ in sel] for _ in range(n_cap)], np.int32)
    with F.AcqEngine(table, F.default_params(**kw)) as eng:
        full_r, full_g = eng.search(np.concatenate(caps), sel=sel, want_grid=True)
        rec, grid = eng.search_aided(np.concatenate(caps), centers, hw, sel=sel, want_grid=True)
        check_against_full(eng, rec, grid, full_g, centers, hw, sel, table)
    thr = np.array([kw["thr_e1b"] if table[s][3] == S.E1B else kw["thr_l1"] for s in sel])
    for c in range(n_cap):
        orec, ogrid = oracle.search(caps[c], table, sel=sel, params=oracle.default_params(**kw), want_grid=True)
        for i in range(len(sel)):
            wlo = window_lo(centers[c, i], hw, lo, hi)
            ow = ogrid[i:i + 1, wlo - lo: wlo - lo + 2 * hw + 1]
            ow_rec = window_pick(ow[0], wlo, sel[i])
            if not ow_rec["snr"] > 0:
                continue   # nothing above zero in the window (a row without a code replica): the record is all zeros
            compare_records(rec[c][i:i + 1], np.array([ow_rec]), ow, wlo, float(thr[i]), ggrid=grid[c][i:i + 1], max_ties=1)


def test_detections_inside_and_outside_the_window(gpu_required):
    table = S.navstar()
    rng = np.random.default_rng(12)
    caps, want = [], []
    for k in range(8):
        sat = int(rng.integers(0, 32))
        dop = int(rng.integers(-18, 19))
        tau = int(rng.integers(0, 4092)) * 4
        caps.append(synth.make_capture(900 + k, 1, table, [(sat, tau, dop * F.BIN_HZ, 50, float(rng.uniform(0, 6)))]))
        want.append((sat, tau // 4, dop))
    hw = 2
    near = np.zeros((8, 32), np.int32)
    far = np.zeros((8, 32), np.int32)
    for k, (sat, _, dop) in enumerate(want):
        near[k, sat] = dop + int(rng.integers(-hw, hw + 1))
        far[k, sat] = dop + 9 if dop < 0 else dop - 9
    with F.AcqEngine(table) as eng:
        rn = eng.search_aided(np.concatenate(caps), near, hw)
        rf = eng.search_aided(np.concatenate(caps), far, hw)
    for k, (sat, lag, dop) in enumerate(want):
        assert (rn[k][sat]["lag"], rn[k][sat]["dop"]) == (lag, dop) and rn[k][sat]["snr"] > 50
        assert rf[k][sat]["dop"] != dop and abs(rf[k][sat]["dop"] - far[k, sat]) <= hw


def test_every_kernel_path(gpu_required):
    """W = 1 on one satellite and one capture (one tile, the capture as the front end's argument, polled records); small
    searches (k_pick_small); 256 captures x 32 satellites (k_best_dop, chunks claimed in k_search_l1_cr)."""
    table = S.navstar()
    caps = np.stack([synth.make_capture(400 + c, 1, table, scenarios.signals("cfg5", c)) for c in range(8)])
    with F.AcqEngine(table) as eng:
        p = eng.params
        sms = eng.device_info()["sm_count"]
        # one tile
        full_r, full_g = eng.search(caps[0], sel=np.array([7], np.int32), want_grid=True)
        n0 = eng.launch_count
        r1 = eng.search_aided(caps[0], np.array([[3]], np.int32), 0, sel=np.array([7], np.int32))
        assert eng.launch_count - n0 == 4   # front end (capture as argument), forward FFT, search, k_pick_small
        _, g1 = eng.search_aided(caps[0], np.array([[3]], np.int32), 0, sel=np.array([7], np.int32), want_grid=True)
        assert g1[0, 0, 0].tobytes() == full_g[0, 0, 3 - p.dop_lo].tobytes()
        assert r1[0, 0].tobytes() == window_pick(g1[0, 0], 3, 7).tobytes()
        # small: 8 captures x 32 satellites, W = 5
        rng = np.random.default_rng(3)
        centers = rng.integers(-25, 26, (8, 32)).astype(np.int32)
        full_r, full_g = eng.search(caps.reshape(-1), want_grid=True)
        rec, grid = eng.search_aided(caps.reshape(-1), centers, 2, want_grid=True)
        check_against_full(eng, rec, grid, full_g, centers, 2, None, table)
        # large: 256 captures x 32 satellites, W = 5 -> 40960 tiles, chunks claimed, best-Doppler pick by k_best_dop
        big = caps[np.arange(256) % 8]
        centers = rng.integers(-25, 26, (256, 32)).astype(np.int32)
        full_r, full_g = eng.search(big.reshape(-1), want_grid=True)
        rec, grid = eng.search_aided(big.reshape(-1), centers, 2, want_grid=True)
        check_against_full(eng, rec, grid, full_g, centers, 2, None, table)
        rec2 = eng.search_aided(big.reshape(-1), centers, 2)
        assert rec2.tobytes() == rec.tobytes()
    plan = _lib.AcqLaunchPlan()
    L = _lib.load()
    assert L.acq_plan_launch(1, 0, 0, 256 * 32 * 5, sms, C.byref(plan)) == 0
    assert plan.kernel == 6 and plan.claims == 1 and plan.n_big > 0   # k_search_l1_cr, chunks claimed


def aided_and_full(table, params, variant, caps, centers, hw, sel=None):
    """Aided search of `caps` on a library variant; with `variant` set its window cells are asserted to be the variant's
    own full grid, to the byte (a forced kernel choice)."""
    with F.AcqEngine(table, params, variant=variant) as eng:
        p = eng.params
        _, full_g = eng.search(caps, sel=sel, want_grid=True)
        rec, grid = eng.search_aided(caps, centers, hw, sel=sel, want_grid=True)
    if variant is not None:
        for c in range(grid.shape[0]):
            for s in range(grid.shape[1]):
                lo = window_lo(centers[c, s], hw, p.dop_lo, p.dop_hi) - p.dop_lo
                assert grid[c, s].tobytes() == full_g[c, s, lo: lo + 2 * hw + 1].tobytes(), (variant, c, s)
    return rec, grid


def test_variant_libraries_agree(gpu_required):
    """The library variants run the aided search on their own kernel choices: each equals its own full search in the
    window bytewise, and the C/A rows equal the product's bytes.  With K = 3, l1_multi_tw runs its full search on
    k_search_l1<true> and its aided search on the product's k_search_l1_multi: the windows still agree."""
    table = scenarios.table("cfg4")
    caps = np.concatenate([synth.make_capture(70 + i, 1, table, scenarios.signals("cfg4", 70 + i)) for i in range(3)])
    sel = np.array([0, 3, 17, 31, 32, 40, 60, 81], np.int32)
    rng = np.random.default_rng(4)
    centers = rng.integers(-24, 25, (3, len(sel))).astype(np.int32)
    out = {}
    for variant in (None, "l1_cta", "l1_multi_tw", "static_tiles", "dyn_tiles", "e1b_cta", "e1b_cluster", "e1b_ldg"):
        out[variant] = aided_and_full(table, F.default_params(), variant, caps, centers, 3, sel)
    ca = np.array([table[s][3] != S.E1B for s in sel])
    for variant in ("l1_cta", "l1_multi_tw", "static_tiles", "dyn_tiles", "e1b_cta", "e1b_cluster", "e1b_ldg"):
        assert out[variant][1][:, ca].tobytes() == out[None][1][:, ca].tobytes(), variant
        assert out[variant][0][:, ca].tobytes() == out[None][0][:, ca].tobytes(), variant
    for variant in ("l1_cta", "l1_multi_tw", "static_tiles", "dyn_tiles"):
        assert out[variant][0].tobytes() == out[None][0].tobytes(), variant
    nav = S.navstar()
    kw = dict(k_noncoh=3, thr_l1=8.0)
    caps3 = np.concatenate([synth.make_capture(80 + i, 3, nav, scenarios.signals("cfg1", 80 + i)) for i in range(2)])
    centers3 = rng.integers(-24, 25, (2, len(nav))).astype(np.int32)
    prod = aided_and_full(nav, F.default_params(**kw), None, caps3, centers3, 3)
    tw = aided_and_full(nav, F.default_params(**kw), "l1_multi_tw", caps3, centers3, 3)
    assert tw[0].tobytes() == prod[0].tobytes() and tw[1].tobytes() == prod[1].tobytes()


def test_device_form_on_a_torch_stream(gpu_required):
    import torch
    table = S.navstar()
    caps = np.concatenate([synth.make_capture(s, 1, table, scenarios.signals("cfg1", s)) for s in (1, 2, 3, 4)])
    rng = np.random.default_rng(5)
    centers = rng.integers(-20, 21, (4, 32)).astype(np.int32)
    with F.AcqEngine(table) as eng:
        host = eng.search_aided(caps, centers, 2)
        full = eng.search(caps)
        d_in = torch.from_numpy(caps).cuda()
        d_c = torch.from_numpy(centers.reshape(-1)).cuda()
        d_out = torch.zeros(4 * 32 * 24, dtype=torch.uint8, device="cuda")
        st = torch.cuda.Stream()
        torch.cuda.synchronize()
        for _ in range(3):
            with torch.cuda.stream(st):
                d_out.zero_()
                eng.search_aided_device(d_in.data_ptr(), d_c.data_ptr(), 2, d_out.data_ptr(), 4, stream_ptr=st.cuda_stream)
            # a host search issued right behind it is ordered after it (shared scratch), and both are right
            assert eng.search(caps).tobytes() == full.tobytes()
            st.synchronize()
            assert d_out.cpu().numpy().tobytes() == host.tobytes()
        sel = np.array([4, 9, 30], np.int32)
        hs = eng.search_aided(caps, centers[:, :3], 1, sel=sel)
        d_out2 = torch.zeros(4 * 3 * 24, dtype=torch.uint8, device="cuda")
        d_c2 = torch.from_numpy(centers[:, :3].reshape(-1).copy()).cuda()
        torch.cuda.synchronize()
        eng.search_aided_device(d_in.data_ptr(), d_c2.data_ptr(), 1, d_out2.data_ptr(), 4, sel=sel)
        assert eng.search_aided(caps, centers, 2).tobytes() == host.tobytes()
        torch.cuda.synchronize()
        assert d_out2.cpu().numpy().tobytes() == hs.tobytes()


def test_refine_after_aided_equals_refine_after_full(gpu_required):
    table = S.reference_table()
    sig = [(2, 4001, 3.3 * F.BIN_HZ, 50, 1.0), (10, 12346, -7.45 * F.BIN_HZ, 48, 2.0), (44, 30003, -6.2 * F.BIN_HZ, 50, 0.4)]
    caps = np.concatenate([synth.make_capture(77 + c, 1, table, sig) for c in range(2)])
    sel = np.array([2, 10, 44, 20, 40], np.int32)
    centers = np.array([[3, -7, -6, 15, 0], [4, -8, -5, -20, 30]], np.int32)
    with F.AcqEngine(table) as eng:
        rec = eng.search_aided(caps, centers, 2, sel=sel)
        fine_aided = eng.refine(rec)
        eng.search(caps, sel=sel)
        fine_full = eng.refine(rec)
    assert fine_aided.tobytes() == fine_full.tobytes()
    assert abs(fine_aided["dop_hz"][0, 0] - 3.3 * F.BIN_HZ) < 0.25 * F.BIN_HZ


def test_alternating_aided_and_full_searches(gpu_required):
    """Aided and full searches alternating on one engine (claimed tiles on both sides, so the tile counters must come back
    to zero after each launch) give the same bytes every time; the argument errors leave the engine usable."""
    table = S.navstar()
    caps = np.concatenate([synth.make_capture(500 + c, 1, table, scenarios.signals("cfg5", c)) for c in range(40)])
    rng = np.random.default_rng(6)
    centers = rng.integers(-20, 21, (40, 32)).astype(np.int32)
    with F.AcqEngine(table) as eng:
        a0 = eng.search_aided(caps, centers, 4)
        f0 = eng.search(caps)
        s0 = eng.search_aided(caps[:8192], centers[:1], 1)
        for _ in range(4):
            assert eng.search_aided(caps, centers, 4).tobytes() == a0.tobytes()
            assert eng.search(caps).tobytes() == f0.tobytes()
            assert eng.search_aided(caps[:8192], centers[:1], 1).tobytes() == s0.tobytes()
        with pytest.raises(F.AcqError) as ei:
            eng.search_aided(caps[:8192], centers[:1], 21)   # W = 43 > n_dop = 41
        assert ei.value.code == -1 and "exceeds n_dop" in str(ei.value)
        with pytest.raises(F.AcqError) as ei:
            eng.search_aided(caps[:8192], centers[:1], -1)
        assert ei.value.code == -1
        out = np.zeros(32, F.RECORD_DTYPE)
        eng.submit(caps[:8192], out)
        with pytest.raises(F.AcqError) as ei:   # a pending submit
            eng.search_aided(caps[:8192], centers[:1], 1)
        assert "pending" in str(ei.value)
        eng.wait()
        assert eng.search_aided(caps, centers, 4).tobytes() == a0.tobytes()


def test_capture_farm_aided_equals_search_aided(gpu_required):
    import torch
    from flydog_sdr_gps_b200 import farm
    table = S.navstar()
    caps = np.stack([synth.make_capture(300 + c, 1, table, scenarios.signals("cfg5", c)) for c in range(5)])
    centers = np.random.default_rng(7).integers(-20, 21, (5, 32)).astype(np.int32)
    with F.AcqEngine(table) as eng:
        want = eng.search_aided(caps.reshape(-1), centers, 2)
        st = torch.cuda.Stream()
        with torch.cuda.stream(st):
            f = farm.CaptureFarm(eng, 5, 8192, 32, half_width=2)
            f.load(caps, dop_center=centers)
            got = f.search().copy()
            f.search_resident()
            st.synchronize()
            res = f.d_all.cpu().numpy().view(F.RECORD_DTYPE).reshape(5, 32)
    assert got.tobytes() == want.tobytes() and res.tobytes() == want.tobytes()
