"""GPU suite (-m gpu) of the hand-off of coherent records (acq_refine_coherent*, acq_profile_coherent*): M = 1 bytes
against acq_refine / acq_profile after acq_search, M > 1 profiles bitwise against the search's own cells and against the
float64 reference, M > 1 refinement against tests/coherent_handoff_ref.py, host and device forms, min_snr and marker
rows, refusals, accuracy on injected signals, the farm, and the engine's lifetime."""
import numpy as np
import pytest

import flydog_sdr_gps_b200 as F
from flydog_sdr_gps_b200 import synth
from flydog_sdr_gps_b200 import sats as S

from coherent_handoff_ref import CoherentHandoffRef, check_fine_coherent
from profile_ref import peak2_of
from search_ref import NOISE_RTOL, PEAK_RTOL, PROFILE_TAU, Worst, check_profile
from test_gpu_coherent import _m1_shape

pytestmark = pytest.mark.gpu
BIN = F.BIN_HZ
L = F.LAGS_L1


def _dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a).reshape(-1).view(np.uint8).copy()).cuda()


def _zeros(nbytes):
    import torch
    return torch.zeros(max(int(nbytes), 1), dtype=torch.uint8, device="cuda")


def _host(t, dtype):
    return t.cpu().numpy().view(dtype)


@pytest.mark.parametrize("name", ["full_bins_k1", "half_bins_k4", "circular_wrap_k4", "two_bit_k1_half_bins", "sbas_row_k2"])
def test_m1_is_refine_and_profile(gpu_required, name):
    """M = 1: refine_coherent / profile_coherent (and its lag profiles) after search_coherent(.., 1) are the bytes of
    refine / profile after search on the same engine and bytes."""
    table, kw, K, bits, sel = _m1_shape(name)
    sig = [(7, 4445, 3.3 * BIN, 45, 0.3), (3, 10001, -11.2 * BIN, 44, 1.7), (0, 9, -19.6 * BIN, 46, 2.5)]
    cap = np.concatenate([synth.make_capture(40 + c, K, table, sig, sample_bits=bits) for c in range(2)])
    with F.AcqEngine(table, F.default_params(**kw)) as eng:
        r0 = eng.search(cap, sel=sel)
        f0 = eng.refine(r0)
        p0, q0 = eng.profile(r0, want_profile=True)
        r1 = eng.search_coherent(cap, 1, sel=sel)
        f1 = eng.refine_coherent(r1)
        p1, q1 = eng.profile_coherent(r1, want_profile=True)
    assert r1.tobytes() == r0.tobytes()
    assert f1.tobytes() == f0.tobytes()
    assert p1.tobytes() == p0.tobytes() and q1.tobytes() == q0.tobytes()


def _coh_case(m_coh, groups, half_bin, aided, seed=0):
    """An engine's params, a capture with a signal on sat 9 (sat 14 noise only), and the records / cells of a full or aided
    coherent search of sats [9, 14]."""
    K = m_coh * groups
    nav = S.navstar()
    kw = dict(k_noncoh=K, half_bin=half_bin, dop_lo=-4 * (1 + half_bin), dop_hi=3 * (1 + half_bin))
    Fv = m_coh * (1 + half_bin)
    f = (2 * Fv + 1.3) / Fv * BIN
    cap = synth.make_capture(500 + 7 * K + half_bin + seed, K, nav, [(9, 3003, f, 42, 0.9)])
    return nav, kw, cap, np.array([9, 14], np.int32), Fv


def _search(eng, cap, m_coh, sel, aided):
    if aided:
        centers = np.array([[2 * m_coh * (1 + eng.params.half_bin), -3]], np.int32)
        return eng.search_coherent_aided(cap, m_coh, centers, 4, sel=sel, want_grid=True) + (centers,)
    rec, grid = eng.search_coherent(cap, m_coh, sel=sel, want_grid=True)
    return rec, grid, None


CASES = [(m, g, hb, a) for m in (2, 3, 4, 5) for g, hb, a in ((1, 0, False), (2, 1, False), (2, 0, True))]


@pytest.mark.parametrize("m_coh,groups,half_bin,aided", CASES)
def test_profile_against_search_and_reference(gpu_required, oracle, m_coh, groups, half_bin, aided):
    """M > 1: the profile at the record's lag is rec.peak to the bit and its first maximum is rec.lag; the record's cell
    of the search's grid has that peak and the mean of the row as noise; rows and peak2 / ratio / noise_ex against the
    float64 reference (check_profile's bound, search_ref's tolerances)."""
    nav, kw, cap, sel, Fv = _coh_case(m_coh, groups, half_bin, aided)
    excl = 4
    with F.AcqEngine(nav, F.default_params(**kw)) as eng:
        rec, grid, centers = _search(eng, cap, m_coh, sel, aided)
        out, prof = eng.profile_coherent(rec, excl=excl, want_profile=True)
        p = eng.params
    worst = Worst("profile M = %d" % m_coh)
    lo_full = m_coh * p.dop_lo
    for s, sat in enumerate(sel):
        r, o, row = rec[0, s], out[0, s], prof[s * L:(s + 1) * L]
        assert o["lag2"] >= 0
        assert row[r["lag"]].tobytes() == r["peak"].tobytes()
        assert int(np.argmax(row)) == r["lag"]
        lo = lo_full if centers is None else int(np.clip(centers[0, s] - 4, lo_full, m_coh * p.dop_hi - 8))
        cell = grid[0, s, int(r["dop"]) - lo]
        assert cell["peak"].tobytes() == r["peak"].tobytes() and cell["lag"] == r["lag"]
        assert abs(float(cell["noise"]) / row.astype(np.float64).mean() - 1) < 1e-5
        P = CoherentHandoffRef(oracle, p, cap, nav, int(sat)).power(int(r["dop"]), m_coh)
        check_profile(row, P, worst, "sat %d" % sat)
        peak2, lag2, ratio, noise_ex = peak2_of(P, int(r["lag"]), excl)
        m = P.mean()
        b2 = PROFILE_TAU * np.sqrt(peak2 * m + m * m)   # check_profile's bound at the second peak
        assert o["lag2"] == lag2 or P[o["lag2"]] >= peak2 - 2 * b2, (o, lag2)
        assert abs(o["peak2"] - peak2) <= b2, (o, peak2, b2)
        assert abs(o["ratio"] / ratio - 1) <= PEAK_RTOL + b2 / peak2, (o, ratio)
        assert abs(o["noise_ex"] / noise_ex - 1) <= NOISE_RTOL, (o, noise_ex)
    print(worst)


@pytest.mark.parametrize("m_coh,groups,half_bin,aided", CASES)
def test_refine_against_reference(gpu_required, oracle, m_coh, groups, half_bin, aided):
    """M > 1: the search's records and placed records -- h = M dop_lo and M dop_hi, lags 0 and 4091, the noise row --
    refined within the float64 reference's bound; a search record's refined peak within 1e-5 of rec.peak."""
    nav, kw, cap, sel, Fv = _coh_case(m_coh, groups, half_bin, aided)
    with F.AcqEngine(nav, F.default_params(**kw)) as eng:
        rec, grid, centers = _search(eng, cap, m_coh, sel, aided)
        fine = eng.refine_coherent(rec)
        p = eng.params
        placed = []
        for h, n in ((m_coh * p.dop_lo, 0), (m_coh * p.dop_hi, L - 1), (m_coh * p.dop_lo + 1, 2047), (1, L - 1)):
            r = rec.copy()
            r["dop"], r["lag"] = h, n
            placed.append((r, eng.refine_coherent(r)))
    refs = {int(s): CoherentHandoffRef(oracle, p, cap, nav, int(s)) for s in sel}
    worst = Worst("refine M = %d" % m_coh)
    check_fine_coherent(fine, rec, lambda i, r: refs[int(r["sat"])], m_coh, worst, "search records")
    for f, r in zip(fine.reshape(-1), rec.reshape(-1)):
        assert abs(float(f["peak"]) / float(r["peak"]) - 1) <= 1e-5, (f, r)
    for r, f in placed:
        check_fine_coherent(f, r, lambda i, rr: refs[int(rr["sat"])], m_coh, worst, "placed")
    print(worst)


def test_host_device_min_snr_and_markers(gpu_required):
    """Host form == device form on the engine stream and on a torch stream (profiles too); min_snr marks the rows below it
    (-1) and leaves the others' bytes; bad device records get -2 markers and NaN profiles; a following search waits for
    the hand-off (its spectra are not overwritten under it)."""
    import torch
    nav = S.navstar()
    M, K = 4, 8
    caps = np.concatenate([synth.make_capture(80 + c, K, nav, [(5, 900 + 5 * c, (3.1 - c) * BIN, 40, 0.2)]) for c in range(3)])
    sel = np.array([5, 6, 20], np.int32)
    with F.AcqEngine(nav, F.default_params(k_noncoh=K, half_bin=1)) as eng:
        rec = eng.search_coherent(caps, M, sel=sel)
        fh = eng.refine_coherent(rec)
        ph, qh = eng.profile_coherent(rec, want_profile=True)
        n = rec.size
        d_rec = _dev(rec)
        for st in (None, torch.cuda.Stream()):
            sp = None if st is None else st.cuda_stream
            d_f, d_p, d_q = _zeros(n * 16), _zeros(n * 16), _zeros(n * L * 4)
            torch.cuda.synchronize()
            eng.refine_coherent_device(d_rec.data_ptr(), d_f.data_ptr(), n, stream_ptr=sp)
            eng.profile_coherent_device(d_rec.data_ptr(), d_p.data_ptr(), n, profile_dev=d_q.data_ptr(), stream_ptr=sp)
            torch.cuda.synchronize()
            assert _host(d_f, F.FINE_DTYPE).tobytes() == fh.tobytes()
            assert _host(d_p, F.PEAK2_DTYPE).tobytes() == ph.tobytes() and _host(d_q, np.float32).tobytes() == qh.tobytes()
        thr = float(np.median(rec["snr"]))
        d_f, d_p = _zeros(n * 16), _zeros(n * 16)
        torch.cuda.synchronize()
        eng.refine_coherent_device(d_rec.data_ptr(), d_f.data_ptr(), n, min_snr=thr)
        eng.profile_coherent_device(d_rec.data_ptr(), d_p.data_ptr(), n, min_snr=thr)
        torch.cuda.synchronize()
        fm, pm = _host(d_f, F.FINE_DTYPE), _host(d_p, F.PEAK2_DTYPE)
        keep = rec.reshape(-1)["snr"] >= thr
        assert 0 < keep.sum() < n
        assert (fm["ca_shift"][~keep] == -1).all() and np.isnan(fm["dop_hz"][~keep]).all() and (fm["peak"][~keep] == 0).all()
        assert (pm["lag2"][~keep] == -1).all() and np.isnan(pm["ratio"][~keep]).all()
        assert fm[keep].tobytes() == fh.reshape(-1)[keep].tobytes() and pm[keep].tobytes() == ph.reshape(-1)[keep].tobytes()
        bad = rec.copy().reshape(-1)
        bad["sat"][0] = 6            # not the satellite of slot 0
        bad["lag"][1] = L            # lag out of range
        bad["dop"][2] = M * 2 * eng.params.dop_hi + 2   # beyond M dop_hi
        bad["sat"][3] = 99           # outside the table
        d_bad = _dev(bad)
        d_f, d_p, d_q = _zeros(n * 16), _zeros(n * 16), _zeros(n * L * 4)
        torch.cuda.synchronize()
        eng.refine_coherent_device(d_bad.data_ptr(), d_f.data_ptr(), n)
        eng.profile_coherent_device(d_bad.data_ptr(), d_p.data_ptr(), n, profile_dev=d_q.data_ptr())
        torch.cuda.synchronize()
        fb, pb, qb = _host(d_f, F.FINE_DTYPE), _host(d_p, F.PEAK2_DTYPE), _host(d_q, np.float32).reshape(n, L)
        assert (fb["ca_shift"][:4] == -2).all() and (pb["lag2"][:4] == -2).all() and np.isnan(qb[:4]).all()
        assert fb[4:].tobytes() == fh.reshape(-1)[4:].tobytes() and pb[4:].tobytes() == ph.reshape(-1)[4:].tobytes()
        # ordering: the hand-off on a torch stream, then a search on the engine stream that overwrites the spectra
        st = torch.cuda.Stream()
        other = np.concatenate([synth.make_capture(90 + c, K, nav, []) for c in range(3)])
        d_f = _zeros(n * 16)
        torch.cuda.synchronize()
        for _ in range(3):
            eng.refine_coherent_device(d_rec.data_ptr(), d_f.data_ptr(), n, stream_ptr=st.cuda_stream)
        eng.search_coherent(other, M, sel=sel)
        st.synchronize()
        assert _host(d_f, F.FINE_DTYPE).tobytes() == fh.tobytes()


def test_refusals(gpu_required):
    """ACQ_ERR_ARG with nothing launched and the engine usable afterwards: after a non-coherent search, after no search,
    with an acq_submit pending; a wrong n_records, misaligned pointers, a NaN min_snr, excl out of range."""
    import torch
    nav = S.navstar()
    K, M = 4, 2
    cap = synth.make_capture(33, K, nav, [(2, 4000, 4 * BIN, 46, 1.0)])
    sel = np.array([2, 3], np.int32)
    with F.AcqEngine(nav, F.default_params(k_noncoh=K)) as eng:
        n0 = eng.launch_count
        d_rec, d_out = _zeros(2 * 24 + 64), _zeros(2 * L * 4 + 64)
        torch.cuda.synchronize()
        rec0 = np.zeros(2, F.RECORD_DTYPE)
        rec0["sat"] = sel

        def all_calls(rec, n=2, rp=d_rec.data_ptr(), op=d_out.data_ptr(), min_snr=0.0, excl=4, prof=None):
            return [lambda: eng.refine_coherent(rec), lambda: eng.profile_coherent(rec, excl=excl),
                    lambda: eng.refine_coherent_device(rp, op, n, min_snr=min_snr),
                    lambda: eng.profile_coherent_device(rp, op, n, excl=excl, min_snr=min_snr, profile_dev=prof)]

        def refused(calls, text=None):
            for c in calls:
                with pytest.raises(F.AcqError) as ei:
                    c()
                assert ei.value.code == -1, ei.value
                assert text is None or text in str(ei.value), (text, str(ei.value))

        refused(all_calls(rec0), "coherent")   # no search yet
        assert eng.launch_count == n0
        rec = eng.search(cap, sel=sel)
        n1 = eng.launch_count
        refused(all_calls(rec), "coherent")    # after a non-coherent search
        assert eng.launch_count == n1
        crec = eng.search_coherent(cap, M, sel=sel)
        n2 = eng.launch_count
        d_rec = _dev(crec)
        torch.cuda.synchronize()
        refused(all_calls(crec, n=3, rp=d_rec.data_ptr()) [2:])             # wrong n_records (device forms)
        refused(all_calls(crec[:, :1])[:2])                                   # wrong n_records (host forms)
        refused(all_calls(crec, rp=d_rec.data_ptr() + 2)[2:])                 # rec_dev misaligned
        refused(all_calls(crec, rp=d_rec.data_ptr(), op=d_out.data_ptr() + 4)[2:])   # out_dev misaligned
        refused(all_calls(crec, rp=d_rec.data_ptr(), prof=d_out.data_ptr() + 2)[3:])  # profile_dev misaligned
        refused(all_calls(crec, rp=d_rec.data_ptr(), min_snr=float("nan"))[2:], "NaN")
        for excl in (-1, L // 2):
            refused([c for i, c in enumerate(all_calls(crec, rp=d_rec.data_ptr(), excl=excl)) if i in (1, 3)], "excl")
        assert eng.launch_count == n2
        fine = eng.refine_coherent(crec)                   # still usable
        assert (fine["ca_shift"] >= 0).all()
        out = np.zeros(2, F.RECORD_DTYPE)
        eng.submit(cap, out, sel=sel)
        refused(all_calls(crec, rp=d_rec.data_ptr()), "pending")
        eng.wait()
        n3 = eng.launch_count
        refused(all_calls(out.reshape(1, 2), rp=d_rec.data_ptr()), "coherent")   # acq_submit is a non-coherent search
        assert eng.launch_count == n3
        assert eng.refine(out.reshape(1, 2)).shape == (1, 2)


# Accuracy of the hand-off: the cfg2 shape (tools/coherent_bench.CFG2: K = 20, half-bins, +-80) at M = 4, 64 captures of
# one PRN at 33 dB-Hz with a random code phase (any FS sample, so the truth lies between lags) and a Doppler uniform in
# +-9 kHz.  Over the found rows (lag within +-1, Doppler within one coherent step).  The bounds come from one run on an
# NVIDIA B200 (1000 W power limit), profiles/coherent_handoff_bench_b200.json, same workload at M = 4 with 128
# captures: median Doppler error refined / grid-only 3.7 / 7.1 Hz at 31 dB-Hz and 2.2 / 7.8 Hz at 35 dB-Hz; median
# code-phase error 0.61 / 1.0 and 0.38 / 1.0 FS samples; found 0.88 and 1.0.  This test passed at these bounds in the
# same run.
ACC_CN0 = 33.0


def _bench():
    import os
    import sys
    tools = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools")
    if tools not in sys.path:
        sys.path.insert(0, tools)
    import coherent_handoff_bench
    return coherent_handoff_bench


def test_accuracy_beats_the_grid(gpu_required):
    import torch
    B = _bench()
    caps, tau, f = B.handoff_set(F, S, synth, torch, 4242, 64, ACC_CN0)
    with F.AcqEngine(S.navstar(), F.default_params(**B.CFG2)) as eng:
        rec = eng.search_coherent(caps, 4, sel=[7])[:, 0]
        fine = eng.refine_coherent(rec.reshape(-1, 1))[:, 0]
        acc = B.accuracy(F, eng, rec, fine, 4, tau, f)
    print("accuracy", acc)
    assert acc["found"] >= 0.8, acc
    assert acc["dop_hz_refined"]["median"] < 0.6 * acc["dop_hz_grid"]["median"], acc
    assert acc["code_fs_refined"]["median"] < 0.8 * acc["code_fs_grid"]["median"], acc


def test_capture_farm(gpu_required):
    """CaptureFarm(..., m_coh) and the aided coherent farm: refine_coherent() / profile_coherent() are the engine's
    device forms' bytes; a non-coherent farm raises ValueError."""
    import torch
    from flydog_sdr_gps_b200 import farm
    nav = S.navstar()
    M, K = 2, 4
    caps = np.stack([synth.make_capture(300 + c, K, nav, [(c, 4 * (500 + c), (c - 2.5) * BIN, 45, 0.3)]) for c in range(5)])
    centers = np.random.default_rng(7).integers(-40, 41, (5, 32)).astype(np.int32)
    with F.AcqEngine(nav, F.default_params(k_noncoh=K)) as eng:
        st = torch.cuda.Stream()
        with torch.cuda.stream(st):
            for kw, load_kw in ((dict(m_coh=M), {}), (dict(m_coh=M, half_width=3), dict(dop_center=centers))):
                fm = farm.CaptureFarm(eng, 5, K * 8192, 32, **kw)
                fm.load(caps, **load_kw)
                rec = fm.search().copy()
                fine = fm.refine_coherent().copy()
                pk = fm.profile_coherent(excl=3).copy()
                fine_m = fm.refine_coherent(min_snr=float(np.median(rec["snr"]))).copy()
                d_rec = _dev(rec)
                d_f, d_p = _zeros(rec.size * 16), _zeros(rec.size * 16)
                st.synchronize()
                eng.refine_coherent_device(d_rec.data_ptr(), d_f.data_ptr(), rec.size, stream_ptr=st.cuda_stream)
                eng.profile_coherent_device(d_rec.data_ptr(), d_p.data_ptr(), rec.size, excl=3, stream_ptr=st.cuda_stream)
                st.synchronize()
                assert fine.tobytes() == _host(d_f, F.FINE_DTYPE).tobytes()
                assert pk.tobytes() == _host(d_p, F.PEAK2_DTYPE).tobytes()
                assert ((fine_m["ca_shift"] == -1) == (rec["snr"] < np.median(rec["snr"]))).all()
            plain = farm.CaptureFarm(eng, 5, K * 8192, 32)
            plain.load(caps)
            plain.search()
            for call in (plain.refine_coherent, plain.profile_coherent, plain.refine_coherent_resident,
                         plain.profile_coherent_resident):
                with pytest.raises(ValueError):
                    call()


def test_engine_lifetime(gpu_required):
    """acq_create / coherent search / refine_coherent / profile_coherent (host and device) / acq_destroy, thirty times:
    device memory returns to where it was."""
    import torch
    nav = S.navstar()
    cap = synth.make_capture(12, 4, nav, [(2, 4000, 4 * BIN, 48, 1.0)])
    d_in = _dev(cap)
    n = 32
    d_rec, d_f, d_p, d_q = _zeros(n * 24), _zeros(n * 16), _zeros(n * 16), _zeros(n * L * 4)
    torch.cuda.synchronize()

    def cycle():
        with F.AcqEngine(nav, F.default_params(k_noncoh=4, half_bin=1)) as eng:
            r = eng.search_coherent(cap, 2)
            f = eng.refine_coherent(r)
            pk, q = eng.profile_coherent(r, want_profile=True)
            eng.search_coherent_device(d_in.data_ptr(), 2, d_rec.data_ptr(), 1)
            eng.refine_coherent_device(d_rec.data_ptr(), d_f.data_ptr(), n)
            eng.profile_coherent_device(d_rec.data_ptr(), d_p.data_ptr(), n, profile_dev=d_q.data_ptr())
            torch.cuda.synchronize()
            assert _host(d_f, F.FINE_DTYPE).tobytes() == f.tobytes() and _host(d_q, np.float32).tobytes() == q.tobytes()
    cycle()
    torch.cuda.synchronize()
    free0 = torch.cuda.mem_get_info()[0]
    for _ in range(30):
        cycle()
    torch.cuda.synchronize()
    assert free0 - torch.cuda.mem_get_info()[0] < (32 << 20)
