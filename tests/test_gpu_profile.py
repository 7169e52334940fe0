"""GPU suite (-m gpu) of the peak-quality profile (acq_profile / acq_profile_device): the lag profile against the oracle's
Correlate restatement and the second-peak reduction against the same reduction in Python, a duplicated code, host
against device form after full and aided searches, the markers, ordering across streams, repeatability and the farms."""
import numpy as np
import pytest

import flydog_sdr_gps_b200 as F
from flydog_sdr_gps_b200 import scenarios, synth
from flydog_sdr_gps_b200 import sats as S

from parity import RTOL
from profile_ref import circular_distance, orc_profile, peak2_of

pytestmark = pytest.mark.gpu

EXCL = 4
SIG_REF = [(2, 4001, 3.3 * F.BIN_HZ, 50, 1.0), (10, 12346, -7.45 * F.BIN_HZ, 48, 2.0), (44, 30003, -6.2 * F.BIN_HZ, 50, 0.4)]
SEL_REF = np.array([2, 10, 44, 20, 58], np.int32)   # C/A rows 2, 10, 20; E1B rows 44, 58


def _ref_caps(n, blocks=1):
    return np.concatenate([synth.make_capture(77 + c, blocks, S.reference_table(), SIG_REF) for c in range(n)])


def _shape(name):
    """(table, params keywords, one capture, sel) of the engine shapes compared with the oracle."""
    nav = S.navstar()
    if name in ("cfg1", "cfg3", "cfg4"):
        sel = {"cfg1": None, "cfg3": np.arange(0, 50, 7, dtype=np.int32),
               "cfg4": np.array([0, 3, 9, 17, 31, 32, 40, 51, 70, 81], np.int32)}[name]
        t = scenarios.table(name)
        return t, scenarios.params_kw(name), synth.make_capture(41, 1, t, scenarios.signals(name, 3)), sel
    if name == "cfg2":
        sig = scenarios.signals("cfg2", 2)
        return nav, scenarios.params_kw("cfg2"), synth.make_capture(42, 20, nav, sig), np.array([s[0] for s in sig[:3]] + [30], np.int32)
    if name == "k4":
        return nav, dict(k_noncoh=4), synth.make_capture(43, 4, nav, scenarios.signals("cfg1", 4)), np.arange(0, 32, 3, dtype=np.int32)
    if name == "code_doppler":
        kw = dict(k_noncoh=5, half_bin=1, dop_lo=-60, dop_hi=60, code_doppler=1, thr_l1=4.0)
        sig = [(4, 9000, 7000.0, 44, 0.2), (11, 300, -5100.0, 44, 1.0)]
        return nav, kw, synth.make_capture(44, 5, nav, sig, code_doppler=True), np.array([4, 11, 19], np.int32)
    if name == "half_bin":
        return nav, dict(half_bin=1, dop_lo=-41, dop_hi=40), synth.make_capture(45, 1, nav, scenarios.signals("cfg1", 5)), None
    if name == "sample_bits_2":
        return nav, dict(sample_bits=2), synth.make_capture(46, 1, nav, scenarios.signals("cfg1", 6), sample_bits=2), None
    if name == "circular":
        return S.reference_table(), dict(wrap_mode=F.WRAP_CIRCULAR), _ref_caps(1), SEL_REF
    if name == "cfg3_k4":   # E1B with K > 1: the running block sums in shared memory
        t = scenarios.table("cfg3_k4")
        kw = scenarios.params_kw("cfg3_k4")
        return t, kw, synth.make_capture(47, kw["k_noncoh"], t, scenarios.signals("cfg3_k4", 1)), np.arange(0, 50, 9, dtype=np.int32)
    if name == "mixed_k3_half_bins":   # C/A and E1B slots interleaved, K > 1: both launches, profile offsets across types
        return S.reference_table(), dict(k_noncoh=3, half_bin=1, dop_lo=-30, dop_hi=30), _ref_caps(1, 3), SEL_REF
    raise KeyError(name)


SHAPES = ["cfg1", "cfg2", "cfg3", "cfg4", "k4", "code_doppler", "half_bin", "sample_bits_2", "circular", "cfg3_k4",
          "mixed_k3_half_bins"]


def _dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a).reshape(-1).view(np.uint8).copy()).cuda()


def _profile_dev(eng, rec_dev, shape, n_prof, detected_only=False, stream=None, excl=EXCL):
    """acq_profile_device on the engine stream (stream None) or a torch stream; waits; returns (rows, profile)."""
    import torch
    n = int(np.prod(shape))
    out = torch.empty(n * 16, dtype=torch.uint8, device="cuda")
    prof = torch.empty(max(n_prof, 1), dtype=torch.float32, device="cuda")
    if stream is None:
        eng.profile_device(rec_dev.data_ptr(), out.data_ptr(), n, excl=excl, detected_only=detected_only,
                           profile_dev=prof.data_ptr())
        torch.cuda.synchronize()
    else:
        with torch.cuda.stream(stream):
            eng.profile_device(rec_dev.data_ptr(), out.data_ptr(), n, excl=excl, detected_only=detected_only,
                               profile_dev=prof.data_ptr(), stream_ptr=stream.cuda_stream)
        stream.synchronize()
    return out.cpu().numpy().view(F.PEAK2_DTYPE).reshape(shape), prof.cpu().numpy()[:n_prof]


def _n_prof(eng, rec):
    return int(eng.lags_of(rec["sat"].reshape(-1)).sum())


@pytest.mark.parametrize("name", SHAPES)
def test_profile_matches_oracle(gpu_required, oracle, name):
    """Every row's lag profile against orc_profile within the parity tolerance; the profile at the record's lag is the
    record's peak to the bit and its first maximum is the record's lag; peak2 / lag2 / noise_ex against the Python
    reduction of the oracle's profile (lags within RTOL of the oracle's second peak count as ties) and against the
    GPU's own profile."""
    table, kw, cap, sel = _shape(name)
    oprm = oracle.default_params(**kw)
    with F.AcqEngine(table, F.default_params(**kw)) as eng:
        rec = eng.search(cap, sel=sel)[0]
        pk, prof = eng.profile(rec, excl=EXCL, want_profile=True)
        off = eng.profile_offsets(1, sel)
    assert prof.size == off[-1]
    for i, r in enumerate(rec):
        row = prof[off[i]:off[i + 1]]
        lag = int(r["lag"])
        assert row[lag] == r["peak"], (i, row[lag], r["peak"])
        assert int(np.argmax(row)) == lag
        P = orc_profile(oracle, oprm, cap, table, int(r["sat"]), int(r["dop"]))
        assert row.size == P.size
        assert np.allclose(row, P, rtol=RTOL, atol=RTOL * P.mean()), (i, np.max(np.abs(row - P)) / P.mean())
        # the kernel's reduction of its own profile
        out = circular_distance(row.size, lag) > EXCL
        g = pk[i]
        assert g["peak2"] == row[out].max() and g["lag2"] == np.nonzero(out & (row == row[out].max()))[0][0]
        assert g["ratio"] == np.float32(row[lag]) / np.float32(g["peak2"])
        assert abs(g["noise_ex"] - row[out].astype(np.float64).mean()) <= 1e-5 * g["noise_ex"]
        # ... against the oracle's
        o_peak2, o_lag2, o_ratio, o_noise = peak2_of(P, lag, EXCL)
        assert abs(g["peak2"] - o_peak2) <= RTOL * o_peak2
        assert g["lag2"] == o_lag2 or (out[g["lag2"]] and P[g["lag2"]] >= (1 - RTOL) * o_peak2), (i, g["lag2"], o_lag2)
        assert abs(g["ratio"] - o_ratio) <= 2 * RTOL * o_ratio
        assert abs(g["noise_ex"] - o_noise) <= RTOL * o_noise


def test_duplicate_code(gpu_required):
    """One PRN twice, 1000 lags apart, amplitudes 1 and 0.5: lag2 lands on the weak copy and ratio is within 20 % of the
    injected power ratio 4; the same strong signal alone has a much larger ratio."""
    nav = S.navstar()
    tau, f = 8000, 6 * F.BIN_HZ
    strong, weak = (7, tau, f, 53.0, 0.4), (7, tau + 4000, f, 53.0 + 20 * np.log10(0.5), 1.9)
    dup = synth.make_capture(90, 1, nav, [strong, weak])
    alone = synth.make_capture(90, 1, nav, [strong])
    weak_only = synth.make_capture(91, 1, nav, [weak])
    sel = np.array([7], np.int32)
    with F.AcqEngine(nav) as eng:
        want_lag2 = int(eng.search(weak_only, sel=sel)[0, 0]["lag"])
        rec = eng.search(dup, sel=sel)
        pk = eng.profile(rec)[0, 0]
        clean = eng.profile(eng.search(alone, sel=sel))[0, 0]
    assert abs(int(circular_distance(F.LAGS_L1, int(rec[0, 0]["lag"]))[want_lag2]) - 1000) <= 1
    assert abs(int(pk["lag2"]) - want_lag2) <= 1, (pk, want_lag2)
    assert abs(pk["ratio"] / 4.0 - 1) <= 0.2, pk
    assert clean["ratio"] > 4 * pk["ratio"], (clean, pk)


@pytest.mark.parametrize("K", [1, 3])
def test_host_and_device_forms_agree(gpu_required, K):
    """acq_profile (host) against acq_profile_device on the same records -- engine stream and a torch stream, after a
    host search, a device search, and aided searches of both paths -- rows and profiles equal to the byte; a repeated
    call gives the same bytes.  C/A and E1B slots in one search, with one block and with three."""
    import torch
    table = S.reference_table()
    caps = _ref_caps(3, K)
    centers = np.array([[3, -7, -6, 20, -20], [-25, 19, 40, 0, 2 ** 31 - 1], [0, 0, 0, 0, 0]], np.int32)
    st = torch.cuda.Stream()
    with F.AcqEngine(table, F.default_params(k_noncoh=K)) as eng:
        rec = eng.search(caps, sel=SEL_REF)
        want, want_p = eng.profile(rec, want_profile=True)
        again, again_p = eng.profile(rec, want_profile=True)
        assert again.tobytes() == want.tobytes() and again_p.tobytes() == want_p.tobytes()
        assert (want["lag2"] >= 0).all() and want_p.size == 3 * (3 * F.LAGS_L1 + 2 * F.LAGS_E1B)
        n_prof = want_p.size
        rec_dev, d_in = _dev(rec), _dev(caps)
        torch.cuda.synchronize()
        for s in (None, st, None):
            got, got_p = _profile_dev(eng, rec_dev, rec.shape, n_prof, stream=s)
            assert got.tobytes() == want.tobytes() and got_p.tobytes() == want_p.tobytes()
        d_rec = torch.zeros(rec.size * 24, dtype=torch.uint8, device="cuda")
        eng.search_device(d_in.data_ptr(), d_rec.data_ptr(), 3, sel=SEL_REF)
        got, got_p = _profile_dev(eng, d_rec, rec.shape, n_prof)
        assert got.tobytes() == want.tobytes() and got_p.tobytes() == want_p.tobytes()
        # aided
        rec_a = eng.search_aided(caps, centers, 2, sel=SEL_REF)
        want_a, want_ap = eng.profile(rec_a, want_profile=True)
        d_c = torch.from_numpy(centers.reshape(-1)).cuda()
        torch.cuda.synchronize()
        with torch.cuda.stream(st):
            eng.search_aided_device(d_in.data_ptr(), d_c.data_ptr(), 2, d_rec.data_ptr(), 3, sel=SEL_REF,
                                    stream_ptr=st.cuda_stream)
        got, got_p = _profile_dev(eng, d_rec, rec.shape, n_prof)
        assert d_rec.cpu().numpy().tobytes() == rec_a.tobytes()
        assert got.tobytes() == want_a.tobytes() and got_p.tobytes() == want_ap.tobytes()


def _assert_marker(pk, code):
    assert np.isnan(pk["peak2"]).all() and np.isnan(pk["ratio"]).all() and np.isnan(pk["noise_ex"]).all()
    assert (pk["lag2"] == code).all()


def test_markers(gpu_required):
    """ACQ_PROFILE_DETECTED: detected rows keep the bytes of the all-rows output (row and profile), the others carry
    lag2 = -1 and a NaN profile row.  Records that fail a check carry lag2 = -2 and a NaN profile row, also under
    ACQ_PROFILE_DETECTED; every other row keeps its bytes."""
    import torch
    table = S.reference_table()
    caps = _ref_caps(3)
    with F.AcqEngine(table, F.default_params(thr_e1b=30.0, dop_lo=-12, dop_hi=-1)) as eng:
        rec = eng.search(caps, sel=SEL_REF)
        n_prof = _n_prof(eng, rec)
        off = eng.profile_offsets(3, SEL_REF)
        rec_dev = _dev(rec)
        torch.cuda.synchronize()
        full, full_p = _profile_dev(eng, rec_dev, rec.shape, n_prof)
        for _ in range(2):
            n0 = eng.launch_count
            det, det_p = _profile_dev(eng, rec_dev, rec.shape, n_prof, detected_only=True)
            assert eng.launch_count - n0 == 2   # the C/A and the E1B rows
        mask = eng.detected(rec).reshape(-1)
        bad = rec.copy().reshape(-1)
        edits = {0: ("sat", -1), 1: ("sat", len(table)), 2: ("sat", int(SEL_REF[4])), 5: ("lag", -1),
                 7: ("lag", F.LAGS_E1B), 8: ("dop", 0), 11: ("dop", 10 ** 6)}
        for row, (field, value) in edits.items():
            bad[row][field] = value
        bad_dev = _dev(bad)
        torch.cuda.synchronize()
        got, got_p = _profile_dev(eng, bad_dev, (rec.size,), n_prof)
        got_d, got_dp = _profile_dev(eng, bad_dev, (rec.size,), n_prof, detected_only=True)
    assert mask.any() and (~mask).any()
    full, det = full.reshape(-1), det.reshape(-1)

    def rows(p, idx):
        return np.concatenate([p[off[i]:off[i + 1]] for i in idx]) if len(idx) else np.zeros(0, np.float32)
    on, off_rows = np.nonzero(mask)[0], np.nonzero(~mask)[0]
    assert det[on].tobytes() == full[on].tobytes() and rows(det_p, on).tobytes() == rows(full_p, on).tobytes()
    _assert_marker(det[off_rows], -1)
    assert np.isnan(rows(det_p, off_rows)).all()
    marked = np.array(sorted(edits))
    kept = np.setdiff1d(np.arange(rec.size), marked)
    for g, gp in ((got, got_p), (got_d, got_dp)):
        _assert_marker(g[marked], -2)
        assert np.isnan(rows(gp, marked)).all()
    assert got[kept].tobytes() == full[kept].tobytes() and rows(got_p, kept).tobytes() == rows(full_p, kept).tobytes()


def test_ordering_and_arguments(gpu_required):
    import torch
    table = S.navstar()
    caps_a = np.concatenate([synth.make_capture(700 + c, 1, table, scenarios.signals("cfg5", c)) for c in range(4)])
    caps_b = np.concatenate([synth.make_capture(800 + c, 1, table, scenarios.signals("cfg5", 10 + c)) for c in range(6)])
    with F.AcqEngine(table) as eng:
        rec_a = eng.search(caps_a)
        pk_a = eng.profile(rec_a)
        rec_b = eng.search(caps_b)
    rows = rec_a.size
    d_rec = torch.zeros(rows * 24 + 16, dtype=torch.uint8, device="cuda")
    d_out = torch.zeros(rows * 16 + 16, dtype=torch.uint8, device="cuda")
    d_prof = torch.zeros(rows * F.LAGS_L1 + 4, dtype=torch.float32, device="cuda")
    d_in = _dev(caps_a)
    torch.cuda.synchronize()
    with F.AcqEngine(table) as eng:
        def profile(n=rows, rec_off=0, out_off=0, excl=EXCL, prof_off=None):
            eng.profile_device(d_rec.data_ptr() + rec_off, d_out.data_ptr() + out_off, n, excl=excl,
                               profile_dev=None if prof_off is None else d_prof.data_ptr() + prof_off)

        with pytest.raises(F.AcqError, match="no search"):
            profile()
        with pytest.raises(F.AcqError, match="no completed host-path search"):
            eng.profile(rec_a)
        out = np.zeros((4, 32), F.RECORD_DTYPE)
        eng.submit(caps_a, out)
        with pytest.raises(F.AcqError, match="pending"):
            profile()
        with pytest.raises(F.AcqError, match="pending"):
            eng.profile(rec_a)
        eng.wait()
        with pytest.raises(F.AcqError, match="n_records"):
            profile(rows - 1)
        with pytest.raises(F.AcqError, match="n_records"):
            eng.profile(rec_a[:3])
        for excl in (F.LAGS_L1 // 2, 10 ** 6):
            with pytest.raises(F.AcqError, match="excl"):
                profile(excl=excl)
            with pytest.raises(F.AcqError, match="excl"):
                eng.profile(rec_a, excl=excl)
        bad = rec_a.copy()
        bad[1, 3]["lag"] = F.LAGS_L1
        with pytest.raises(F.AcqError, match="lag"):
            eng.profile(bad)
        with pytest.raises(F.AcqError, match="16-byte"):
            profile(out_off=8)
        with pytest.raises(F.AcqError, match="4-byte"):
            profile(rec_off=2)
        with pytest.raises(F.AcqError, match="4-byte"):
            profile(prof_off=2)   # bytes: a float pointer off by two bytes
        assert eng.profile(rec_a, excl=F.LAGS_L1 // 2 - 1)["lag2"].min() >= 0   # the largest excl is accepted
        # device search on stream A, profile on stream B, a host search of other captures issued at once: the profile
        # waits for the search, and the next search waits for the profile
        sa, sb = torch.cuda.Stream(), torch.cuda.Stream()
        d_out.zero_()
        torch.cuda.synchronize()
        with torch.cuda.stream(sa):
            eng.search_device(d_in.data_ptr(), d_rec.data_ptr(), 4, stream_ptr=sa.cuda_stream)
        with torch.cuda.stream(sb):
            eng.profile_device(d_rec.data_ptr(), d_out.data_ptr(), rows, stream_ptr=sb.cuda_stream)
        assert eng.search(caps_b).tobytes() == rec_b.tobytes()
        sb.synchronize()
        assert d_out[:rows * 16].cpu().numpy().tobytes() == pk_a.tobytes()
        # host acq_profile after a device search is refused
        eng.search_device(d_in.data_ptr(), d_rec.data_ptr(), 4)
        with pytest.raises(F.AcqError):
            eng.profile(rec_a)
        torch.cuda.synchronize()


def test_excl_bound_follows_the_searched_types(gpu_required):
    """excl < L_min / 2 with L_min the smallest L of the searched satellites: an E1B-only search accepts excl up to
    8183 (refused for a search with a C/A slot from 2046 on), in both forms."""
    import torch
    t3 = scenarios.table("cfg3")
    cap = synth.make_capture(49, 1, t3, scenarios.signals("cfg3", 2))
    sel = np.array([0, 7, 21], np.int32)
    with F.AcqEngine(t3) as eng:
        rec = eng.search(cap, sel=sel)
        rec_dev = _dev(rec)
        out = torch.zeros(rec.size * 16, dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()
        for excl in (F.LAGS_L1 // 2, F.LAGS_E1B // 2 - 1):
            pk = eng.profile(rec, excl=excl)
            assert (pk["lag2"] >= 0).all()
            eng.profile_device(rec_dev.data_ptr(), out.data_ptr(), rec.size, excl=excl)
            torch.cuda.synchronize()
            assert out.cpu().numpy().tobytes() == pk.tobytes()
            d = circular_distance(F.LAGS_E1B, int(rec[0, 0]["lag"]))[pk[0, 0]["lag2"]]
            assert d > excl
        for excl in (F.LAGS_E1B // 2, 10 ** 6):
            with pytest.raises(F.AcqError, match="excl"):
                eng.profile(rec, excl=excl)
            with pytest.raises(F.AcqError, match="excl"):
                eng.profile_device(rec_dev.data_ptr(), out.data_ptr(), rec.size, excl=excl)
    with F.AcqEngine(S.reference_table()) as eng:   # a C/A slot among E1B ones: L_min = 4092
        rec = eng.search(_ref_caps(1), sel=SEL_REF)
        with pytest.raises(F.AcqError, match="excl"):
            eng.profile(rec, excl=F.LAGS_L1 // 2)
        assert (eng.profile(rec, excl=F.LAGS_L1 // 2 - 1)["lag2"] >= 0).all()


def test_host_profile_buffer_is_released(gpu_required):
    """The host form's lag-profile buffer (256 MiB here) is freed before the call returns."""
    import torch
    nav = S.navstar()
    caps = np.concatenate([synth.make_capture(900 + c, 1, nav, scenarios.signals("cfg5", c)) for c in range(512)])
    with F.AcqEngine(nav) as eng:
        rec = eng.search(caps)
        eng.profile(rec)
        torch.cuda.synchronize()
        free0 = torch.cuda.mem_get_info()[0]
        pk, prof = eng.profile(rec, want_profile=True)
        torch.cuda.synchronize()
        assert prof.size == 512 * 32 * F.LAGS_L1 and (pk["lag2"] >= 0).all()
        assert free0 - torch.cuda.mem_get_info()[0] < (32 << 20)


def test_farms_on_one_gpu(gpu_required):
    """CaptureFarm (full, and aided with half_width 2) and SatFarm: profile() equals acq_profile after a host search of
    the same captures; profile() with its default detected_only marks the undetected rows."""
    import torch
    from flydog_sdr_gps_b200 import farm
    nav = S.navstar()
    caps = np.stack([synth.make_capture(300 + c, 1, nav, scenarios.signals("cfg5", c)) for c in range(5)])
    centers = np.random.default_rng(7).integers(-20, 21, (5, 32)).astype(np.int32)
    ref = S.reference_table()
    cap1 = _ref_caps(1)
    st = torch.cuda.Stream()
    with F.AcqEngine(nav) as eng:
        rec = eng.search(caps.reshape(-1))
        want = eng.profile(rec)
        rec_aided = eng.search_aided(caps.reshape(-1), centers, 2)
        want_aided = eng.profile(rec_aided, excl=8)
        with torch.cuda.stream(st):
            f = farm.CaptureFarm(eng, 5, 8192, 32)
            f.load(caps)
            assert f.search().tobytes() == rec.tobytes()
            got = f.profile(detected_only=False).copy()
            det = f.profile().copy()
            fa = farm.CaptureFarm(eng, 5, 8192, 32, half_width=2)
            fa.load(caps, dop_center=centers)
            assert fa.search().tobytes() == rec_aided.tobytes()
            got_aided = fa.profile(excl=8, detected_only=False).copy()
        mask = eng.detected(rec)
    assert got.shape == (5, 32) and got.tobytes() == want.tobytes()
    assert got_aided.tobytes() == want_aided.tobytes()
    assert det[mask].tobytes() == want[mask].tobytes()
    _assert_marker(det[~mask], -1)
    with F.AcqEngine(ref) as eng:
        want_sat = eng.profile(eng.search(cap1, sel=np.arange(len(ref), dtype=np.int32)))
        with torch.cuda.stream(st):
            fs = farm.SatFarm(eng, len(ref), 8192)
            fs.load(cap1)
            fs.search()
            got_sat = fs.profile(detected_only=False).copy()
    assert got_sat.shape == (len(ref),) and got_sat.tobytes() == want_sat.tobytes()
