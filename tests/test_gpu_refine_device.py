"""GPU suite (-m gpu) of the device-resident refinement (acq_refine_device): the bytes of the host form acq_refine after
a search of either path, the ACQ_REFINE_DETECTED and bad-record markers, the ordering against searches on other streams,
the farms' refine(), and the engine's lifetime."""
import numpy as np
import pytest

import flydog_sdr_gps_b200 as F
from flydog_sdr_gps_b200 import scenarios, synth
from flydog_sdr_gps_b200 import sats as S

pytestmark = pytest.mark.gpu

SIG_REF = [(2, 4001, 3.3 * F.BIN_HZ, 50, 1.0), (10, 12346, -7.45 * F.BIN_HZ, 48, 2.0), (44, 30003, -6.2 * F.BIN_HZ, 50, 0.4)]
SEL_REF = np.array([2, 10, 44, 20, 58], np.int32)   # C/A rows 2, 10, 20; E1B rows 44, 58


def _ref_caps(n):
    return np.concatenate([synth.make_capture(77 + c, 1, S.reference_table(), SIG_REF) for c in range(n)])


def _shape(name):
    """(table, params keywords, captures, sel) of the engine shapes the device form is compared on."""
    nav = S.navstar()
    if name == "reference_k1":
        return S.reference_table(), {}, _ref_caps(2), SEL_REF
    if name == "navstar_k4_half_bins":
        caps = [synth.make_capture(78 + c, 4, nav, [(7, 8002 + c, (4.5 - c) * F.BIN_HZ, 46, 0.5), (12, 100, -3.1 * F.BIN_HZ, 46, 0.1)])
                for c in range(3)]
        return nav, dict(k_noncoh=4, half_bin=1), np.concatenate(caps), None
    if name == "code_doppler":   # cfg2's shape: half-bins, K = 20, 5 shifted copies of every spectrum
        kw = dict(scenarios.params_kw("cfg2"), code_doppler=1)
        cap = synth.make_capture(21, kw["k_noncoh"], nav, scenarios.signals("cfg2", 1), code_doppler=True)
        return nav, kw, cap, np.array([0, 5, 9, 17, 30], np.int32)
    if name == "e1b_k4":
        t3 = scenarios.table("cfg3_k4")
        kw = scenarios.params_kw("cfg3_k4")
        return t3, kw, synth.make_capture(31, kw["k_noncoh"], t3, scenarios.signals("cfg3_k4", 1)), np.arange(0, 50, 5, dtype=np.int32)
    if name == "sample_bits_2":
        caps = [synth.make_capture(60 + c, 1, nav, scenarios.signals("cfg1", c), sample_bits=2) for c in range(2)]
        return nav, dict(sample_bits=2), np.concatenate(caps), None
    if name == "selection":
        caps = [synth.make_capture(500 + c, 1, nav, scenarios.signals("cfg5", c)) for c in range(3)]
        return nav, {}, np.concatenate(caps), np.array([31, 0, 17, 5, 9, 22], np.int32)
    raise KeyError(name)


SHAPES = ["reference_k1", "navstar_k4_half_bins", "code_doppler", "e1b_k4", "sample_bits_2", "selection"]


def _dev(a):
    """A copy of a numpy array on the GPU as uint8 bytes (synchronise before an engine call reads it)."""
    import torch
    return torch.from_numpy(np.ascontiguousarray(a).reshape(-1).view(np.uint8).copy()).cuda()


def _refine_dev(eng, rec_dev, shape, detected_only=False, stream=None):
    """acq_refine_device of rec_dev on the engine stream (stream None) or a torch stream; waits and returns the output.
    Nothing synchronises before the call: the engine orders the refinement behind its search itself."""
    import torch
    n = int(np.prod(shape))
    out = torch.empty(n * 16, dtype=torch.uint8, device="cuda")
    if stream is None:
        eng.refine_device(rec_dev.data_ptr(), out.data_ptr(), n, detected_only=detected_only)
        torch.cuda.synchronize()
    else:
        with torch.cuda.stream(stream):
            eng.refine_device(rec_dev.data_ptr(), out.data_ptr(), n, detected_only=detected_only, stream_ptr=stream.cuda_stream)
        stream.synchronize()
    return out.cpu().numpy().view(F.FINE_DTYPE).reshape(shape)


def _assert_marker(fine, code):
    assert np.isnan(fine["dop_hz"]).all() and np.isnan(fine["code_fs"]).all()
    assert (fine["peak"] == 0).all() and (fine["ca_shift"] == code).all()


@pytest.mark.parametrize("name", SHAPES)
def test_device_form_equals_host_form(gpu_required, name):
    """Host search + acq_refine against acq_refine_device of the same records (engine stream and a torch stream), and
    against acq_search_device + acq_refine_device (the records never leave the GPU): equal to the byte."""
    import torch
    table, kw, caps, sel = _shape(name)
    with F.AcqEngine(table, F.default_params(**kw)) as eng:
        n_cap = caps.size // (eng.k_noncoh * eng.block_bytes)
        rec = eng.search(caps, sel=sel)
        want = eng.refine(rec)
        assert (want["ca_shift"] >= 0).all()
        rec_dev, d_in = _dev(rec), _dev(caps)
        d_rec = torch.zeros(rec.size * 24, dtype=torch.uint8, device="cuda")
        st = torch.cuda.Stream()
        torch.cuda.synchronize()
        assert _refine_dev(eng, rec_dev, rec.shape).tobytes() == want.tobytes()
        assert _refine_dev(eng, rec_dev, rec.shape, stream=st).tobytes() == want.tobytes()
        # device search on the engine stream, refinement right behind it
        eng.search_device(d_in.data_ptr(), d_rec.data_ptr(), n_cap, sel=sel)
        assert _refine_dev(eng, d_rec, rec.shape).tobytes() == want.tobytes()
        assert d_rec.cpu().numpy().tobytes() == rec.tobytes()
        # device search on a torch stream, refinement on the engine stream (ordered by the engine's event)
        d_rec.zero_()
        torch.cuda.synchronize()
        with torch.cuda.stream(st):
            eng.search_device(d_in.data_ptr(), d_rec.data_ptr(), n_cap, sel=sel, stream_ptr=st.cuda_stream)
        assert _refine_dev(eng, d_rec, rec.shape).tobytes() == want.tobytes()


def test_aided_device_equals_aided_host(gpu_required):
    """acq_search_aided_device + acq_refine_device against acq_search_aided + acq_refine, with windows at both edges of
    the range and beyond it."""
    import torch
    table = S.reference_table()
    caps = _ref_caps(2)
    centers = np.array([[3, -7, -6, 20, -20], [-25, 19, 40, 0, 2 ** 31 - 1]], np.int32)
    with F.AcqEngine(table) as eng:
        rec = eng.search_aided(caps, centers, 2, sel=SEL_REF)
        want = eng.refine(rec)
        d_in, d_c = _dev(caps), torch.from_numpy(centers.reshape(-1)).cuda()
        d_rec = torch.zeros(rec.size * 24, dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()
        eng.search_aided_device(d_in.data_ptr(), d_c.data_ptr(), 2, d_rec.data_ptr(), 2, sel=SEL_REF)
        got = _refine_dev(eng, d_rec, rec.shape)
        assert d_rec.cpu().numpy().tobytes() == rec.tobytes()
    assert got.tobytes() == want.tobytes()
    assert abs(got["dop_hz"][0, 0] - 3.3 * F.BIN_HZ) < 0.25 * F.BIN_HZ


def test_detected_only(gpu_required):
    """ACQ_REFINE_DETECTED: detected rows (the threshold of each satellite's type) keep the bytes of the all-rows output,
    the others carry the -1 marker; one kernel launch per call."""
    import torch
    table = S.reference_table()
    caps = _ref_caps(3)
    with F.AcqEngine(table, F.default_params(thr_e1b=30.0)) as eng:
        rec = eng.search(caps, sel=SEL_REF)
        rec_dev = _dev(rec)
        torch.cuda.synchronize()
        full = _refine_dev(eng, rec_dev, rec.shape)
        for _ in range(2):
            n0 = eng.launch_count
            det = _refine_dev(eng, rec_dev, rec.shape, detected_only=True)
            assert eng.launch_count - n0 == 1
        mask = eng.detected(rec)
    assert mask.any() and (~mask).any()
    assert det[mask].tobytes() == full[mask].tobytes()
    _assert_marker(det[~mask], -1)


def test_record_checks(gpu_required):
    """Rows whose record fails a check carry the -2 marker (also under ACQ_REFINE_DETECTED); every other row keeps its
    bytes.  A record of dop 0 with snr 0 is accepted although 0 lies outside this engine's range, as acq_refine accepts it."""
    import torch
    table = S.reference_table()
    caps = _ref_caps(4)
    with F.AcqEngine(table, F.default_params(dop_lo=-12, dop_hi=-1)) as eng:
        rec = eng.search(caps, sel=SEL_REF)
        p = eng.params
        rec_dev = _dev(rec)
        torch.cuda.synchronize()
        full = _refine_dev(eng, rec_dev, rec.shape).reshape(-1)
        bad = rec.copy().reshape(-1)
        # row -> slot = row % 5: slot 0 sat 2 (C/A), 1 sat 10, 2 sat 44 (E1B), 3 sat 20, 4 sat 58 (E1B)
        edits = {0: ("sat", -1), 1: ("sat", len(table)), 2: ("sat", 10 ** 6), 3: ("sat", int(SEL_REF[4])),
                 5: ("lag", -1), 6: ("lag", F.LAGS_L1), 7: ("lag", F.LAGS_E1B), 8: ("dop", p.dop_hi + 1),
                 10: ("dop", p.dop_lo - 1), 11: ("dop", 10 ** 6), 12: ("dop", -(10 ** 6))}
        for row, (field, value) in edits.items():
            bad[row][field] = value
        bad[13]["dop"], bad[13]["snr"] = 0, 0.0   # accepted: the record of a row that never exceeded snr 0
        bad_dev = _dev(bad)
        torch.cuda.synchronize()
        got = _refine_dev(eng, bad_dev, (rec.size,))
        got_det = _refine_dev(eng, bad_dev, (rec.size,), detected_only=True)
        zero = rec.copy().reshape(-1)
        zero[13]["dop"], zero[13]["snr"] = 0, 0.0
        host_zero = eng.refine(zero.reshape(rec.shape)).reshape(-1)
    assert bad[6]["sat"] in (2, 10, 20) and bad[7]["sat"] in (44, 58)
    marked = np.array(sorted(edits))
    kept = np.setdiff1d(np.arange(rec.size), np.append(marked, 13))
    _assert_marker(got[marked], -2)
    _assert_marker(got_det[marked], -2)
    assert got[kept].tobytes() == full[kept].tobytes()
    assert got[13].tobytes() == host_zero[13].tobytes() and got[13]["ca_shift"] >= 0


def test_ordering_and_state(gpu_required):
    import torch
    table = S.navstar()
    caps_a = np.concatenate([synth.make_capture(700 + c, 1, table, scenarios.signals("cfg5", c)) for c in range(4)])
    caps_b = np.concatenate([synth.make_capture(800 + c, 1, table, scenarios.signals("cfg5", 10 + c)) for c in range(6)])
    with F.AcqEngine(table) as eng:
        rec_a = eng.search(caps_a)
        fine_a = eng.refine(rec_a)
        rec_b = eng.search(caps_b)
    rows = rec_a.size
    d_rec = torch.zeros(rows * 24 + 16, dtype=torch.uint8, device="cuda")
    d_out = torch.zeros(rows * 16 + 16, dtype=torch.uint8, device="cuda")
    d_in = _dev(caps_a)
    torch.cuda.synchronize()
    with F.AcqEngine(table) as eng:
        def refine(n=rows, rec_off=0, out_off=0):
            eng.refine_device(d_rec.data_ptr() + rec_off, d_out.data_ptr() + out_off, n)

        with pytest.raises(F.AcqError, match="no search"):
            refine()
        out = np.zeros((4, 32), F.RECORD_DTYPE)
        eng.submit(caps_a, out)
        with pytest.raises(F.AcqError, match="pending"):
            refine()
        eng.wait()
        assert out.tobytes() == rec_a.tobytes()
        with pytest.raises(F.AcqError, match="n_records"):
            refine(rows - 1)
        with pytest.raises(F.AcqError, match="16-byte"):
            refine(out_off=8)
        with pytest.raises(F.AcqError, match="4-byte"):
            refine(rec_off=2)
        # device search on stream A, refinement on stream B, a host search of other captures issued at once: the
        # refinement waits for the search, and the next search waits for the refinement
        sa, sb = torch.cuda.Stream(), torch.cuda.Stream()
        d_out.zero_()
        torch.cuda.synchronize()
        with torch.cuda.stream(sa):
            eng.search_device(d_in.data_ptr(), d_rec.data_ptr(), 4, stream_ptr=sa.cuda_stream)
        with torch.cuda.stream(sb):
            eng.refine_device(d_rec.data_ptr(), d_out.data_ptr(), rows, stream_ptr=sb.cuda_stream)
        assert eng.search(caps_b).tobytes() == rec_b.tobytes()
        sb.synchronize()
        assert d_out[:rows * 16].cpu().numpy().tobytes() == fine_a.tobytes()
        # host acq_refine after a device search is still refused
        eng.search_device(d_in.data_ptr(), d_rec.data_ptr(), 4)
        with pytest.raises(F.AcqError):
            eng.refine(rec_a)
        torch.cuda.synchronize()


def test_farms_on_one_gpu(gpu_required):
    """CaptureFarm (full, and aided with half_width 2) and SatFarm: refine() equals acq_refine after a host search of the
    same captures; refine() with its default detected_only marks the undetected rows."""
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
        want = eng.refine(rec)
        rec_aided = eng.search_aided(caps.reshape(-1), centers, 2)
        want_aided = eng.refine(rec_aided)
        with torch.cuda.stream(st):
            f = farm.CaptureFarm(eng, 5, 8192, 32)
            f.load(caps)
            assert f.search().tobytes() == rec.tobytes()
            got = f.refine(detected_only=False).copy()
            det = f.refine().copy()
            fa = farm.CaptureFarm(eng, 5, 8192, 32, half_width=2)
            fa.load(caps, dop_center=centers)
            assert fa.search().tobytes() == rec_aided.tobytes()
            got_aided = fa.refine(detected_only=False).copy()
        mask = eng.detected(rec)
    assert got.shape == (5, 32) and got.tobytes() == want.tobytes()
    assert got_aided.tobytes() == want_aided.tobytes()
    assert det[mask].tobytes() == want[mask].tobytes()
    _assert_marker(det[~mask], -1)
    with F.AcqEngine(ref) as eng:
        want_sat = eng.refine(eng.search(cap1, sel=np.arange(len(ref), dtype=np.int32)))
        with torch.cuda.stream(st):
            fs = farm.SatFarm(eng, len(ref), 8192)
            fs.load(cap1)
            fs.search()
            got_sat = fs.refine(detected_only=False).copy()
    assert got_sat.shape == (len(ref),) and got_sat.tobytes() == want_sat.tobytes()


def test_engine_lifetime_with_device_refinement(gpu_required):
    """acq_create / host and device searches, each refined on the device / acq_destroy, thirty times: device memory
    returns to where it was."""
    import torch
    table = S.reference_table()
    cap = synth.make_capture(11, 1, table, [(2, 4000, 4 * F.BIN_HZ, 48, 1.0)])
    sel = np.array([2, 40], np.int32)
    d_in = _dev(cap)
    d_rec = torch.zeros(2 * 24, dtype=torch.uint8, device="cuda")
    d_out = torch.zeros(2 * 16, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()

    def cycle():
        with F.AcqEngine(table) as eng:
            r = eng.search(cap, sel=sel)
            eng.search_device(d_in.data_ptr(), d_rec.data_ptr(), 1, sel=sel)
            eng.refine_device(d_rec.data_ptr(), d_out.data_ptr(), 2)
            torch.cuda.synchronize()
            assert d_rec.cpu().numpy().tobytes() == r.tobytes()
            assert d_out.cpu().numpy().tobytes() == eng.refine(eng.search(cap, sel=sel)).tobytes()
    cycle()
    torch.cuda.synchronize()
    free0 = torch.cuda.mem_get_info()[0]
    for _ in range(30):
        cycle()
    torch.cuda.synchronize()
    assert free0 - torch.cuda.mem_get_info()[0] < (32 << 20)
