"""GPU parity suite (-m gpu): the CUDA engine, called through the C ABI, against the CPU oracle on the
same bytes, against the golden vectors of the unmodified reference, and through size-independent
properties at the full BASELINE sizes."""
import ctypes as C

import numpy as np
import pytest

import flydog_sdr_gps_b200 as F
from flydog_sdr_gps_b200 import _lib, scenarios, synth
from flydog_sdr_gps_b200 import sats as S

from parity import RTOL, Margins, compare_records

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ref_engine(gpu_required):
    eng = F.AcqEngine(S.reference_table())
    yield eng
    eng.close()


@pytest.fixture(scope="module")
def nav_engine(gpu_required):
    eng = F.AcqEngine(S.navstar())
    yield eng
    eng.close()


def test_native_library_is_loaded(gpu_required):
    import os
    maps = open("/proc/self/maps").read()
    _lib.load()
    maps = open("/proc/self/maps").read()
    assert os.path.basename(_lib.lib_path()) in maps
    info = F.AcqEngine(S.navstar()[:2]).device_info()
    assert info["sm_count"] >= 100


def test_code_spectra_match_oracle(ref_engine, oracle):
    table = S.reference_table()
    for k in range(len(table)):
        c = ref_engine.code_spectrum(k)
        o = oracle.code_spectrum(table[k])
        assert np.abs(c - o).max() / np.abs(o).max() < 1e-5, k


def test_front_end_bit_exact_and_spectrum(ref_engine, oracle, golden_search, golden_stages):
    cap = golden_search["captures"][0]
    x2, D = ref_engine.capture_spectrum(cap)
    assert np.array_equal(x2, golden_stages["x2"])  # bit-exact vs the unmodified reference
    assert np.abs(D - golden_stages["D"]).max() / np.abs(golden_stages["D"]).max() < 1e-5
    for seed in (1, 2):
        cap = synth.make_capture(seed, 1, S.navstar(), scenarios.signals("cfg1", seed))
        x2, D = ref_engine.capture_spectrum(cap)
        assert np.array_equal(x2, oracle.capture_baseband(cap))
        x2h, Dh = ref_engine.capture_spectrum(cap, 1)
        assert np.array_equal(x2h, oracle.capture_baseband(cap, 1))
        oD = oracle.capture_spectrum(cap, 1)
        assert np.abs(Dh - oD).max() / np.abs(oD).max() < 1e-5


def test_golden_reference_vectors(ref_engine, golden_search):
    """Engine vs the answers of the unmodified reference (all 59 sats, 5 captures): decisions exact."""
    table = S.reference_table()
    caps = golden_search["captures"]
    rec = ref_engine.search(caps.reshape(-1))
    assert rec.shape == (len(caps), len(table))
    for i in range(len(caps)):
        thr = 16.0
        strong = golden_search["snr"][i] >= thr * (1 + RTOL)
        assert np.array_equal(rec[i]["dop"][strong], golden_search["dop"][i][strong])
        assert np.array_equal(rec[i]["lag"][strong], golden_search["lag"][i][strong])
        np.testing.assert_allclose(rec[i]["snr"], golden_search["snr"][i], rtol=RTOL)
        # all sats, not only detected ones, agree unless a numerical tie (none expected on these fixtures)
        assert np.array_equal(rec[i]["dop"], golden_search["dop"][i])
        assert np.array_equal(rec[i]["lag"], golden_search["lag"][i])
        assert np.array_equal(ref_engine.detected(rec[i])[np.abs(golden_search["snr"][i] / thr - 1) > RTOL],
                              (golden_search["snr"][i] >= thr)[np.abs(golden_search["snr"][i] / thr - 1) > RTOL])


@pytest.mark.parametrize("seed", [1, 2, 3, 4, 5, 6])
def test_cfg1_cold_start(nav_engine, oracle, seed):
    table = S.navstar()
    cap = synth.make_capture(seed, 1, table, scenarios.signals("cfg1", seed))
    rec, grid = nav_engine.search(cap, want_grid=True)
    orec, ogrid = oracle.search(cap, table, want_grid=True)
    m = Margins("cfg1 seed %d" % seed)
    compare_records(rec[0], orec, ogrid, -20, 16.0, ggrid=grid[0], margins=m)
    m.report()
    assert (orec["snr"] >= 16).sum() >= 5


@pytest.fixture(scope="module")
def cfg2_engine(gpu_required):
    eng = F.AcqEngine(scenarios.table("cfg2"), F.default_params(**scenarios.params_kw("cfg2")))
    yield eng
    eng.close()


@pytest.mark.parametrize("seed", [1, 2, 3, 4, 5])
def test_cfg2_weak_signal_half_bin_noncoherent(cfg2_engine, oracle, seed):
    """BASELINE configs[1]: 32 PRNs, 161 half-bins, K = 20 blocks, satellites at 30..35 dB-Hz; five captures."""
    table = scenarios.table("cfg2")
    kw = scenarios.params_kw("cfg2")
    sig = scenarios.signals("cfg2", seed)
    cap = synth.make_capture(20 + seed, kw["k_noncoh"], table, sig)
    rec, grid = cfg2_engine.search(cap, want_grid=True)
    orec, ogrid = oracle.search(cap, table, params=oracle.default_params(**kw), want_grid=True)
    m = Margins("cfg2 seed %d" % seed)
    compare_records(rec[0], orec, ogrid, kw["dop_lo"], kw["thr_l1"], ggrid=grid[0], max_ties=1, margins=m)
    m.report()
    found = {int(r["sat"]) for r in rec[0] if r["snr"] >= kw["thr_l1"]}
    strong = {s[0] for s in sig if s[3] >= 33.0}
    assert strong <= found, (strong, found)


@pytest.fixture(scope="module")
def cfg3_engine(gpu_required):
    eng = F.AcqEngine(scenarios.table("cfg3"), F.default_params(**scenarios.params_kw("cfg3")))
    yield eng
    eng.close()


@pytest.mark.parametrize("seed", [1, 2, 3, 4, 5])
def test_cfg3_galileo_e1b(cfg3_engine, oracle, seed):
    """BASELINE configs[2]: all 50 E1-B codes, 81 bins, 16368 lags; five captures."""
    table = scenarios.table("cfg3")
    kw = scenarios.params_kw("cfg3")
    cap = synth.make_capture(30 + seed, 1, table, scenarios.signals("cfg3", seed))
    rec, grid = cfg3_engine.search(cap, want_grid=True)
    orec, ogrid = oracle.search(cap, table, params=oracle.default_params(**kw), want_grid=True)
    m = Margins("cfg3 seed %d" % seed)
    compare_records(rec[0], orec, ogrid, kw["dop_lo"], 16.0, ggrid=grid[0], max_ties=1, margins=m)
    m.report()
    assert (orec["snr"] >= 16).sum() >= 4


@pytest.fixture(scope="module")
def cfg4_engine(gpu_required):
    eng = F.AcqEngine(scenarios.table("cfg4"))
    yield eng
    eng.close()


@pytest.mark.parametrize("seed", [1, 2, 3, 4, 5])
def test_cfg4_combined_sharded_by_satellite(cfg4_engine, oracle, seed):
    """BASELINE configs[3]: 82 PRNs on one capture; sharding the satellite list over 'ranks' gives the same records."""
    table = scenarios.table("cfg4")
    eng = cfg4_engine
    cap = synth.make_capture(40 + seed, 1, table, scenarios.signals("cfg4", seed))
    whole, grid = eng.search(cap, want_grid=True)
    for world in ((2, 4, 8) if seed == 1 else (8,)):
        recs = []
        for rank in range(world):
            lo, hi = scenarios.shard(len(table), rank, world)
            recs.append(eng.search(cap, sel=np.arange(lo, hi, dtype=np.int32))[0])
        assert np.concatenate(recs).tobytes() == whole[0].tobytes()  # bitwise identical however the list is split
    orec, ogrid = oracle.search(cap, table, want_grid=True)
    m = Margins("cfg4 seed %d" % seed)
    compare_records(whole[0], orec, ogrid, -20, 16.0, ggrid=grid[0], max_ties=1, margins=m)
    m.report()


def test_cfg5_receiver_farm_properties(nav_engine, oracle):
    """BASELINE configs[4]: 1024 captures x 32 PRNs in one call (5.5e9 cells).  128 DISTINCT captures -- bench.py's own
    (same seeds, same generator) -- each searched by the oracle too; the other 896 are copies, checked through
    size-independent properties."""
    import bench
    table = S.navstar()
    n_cap, distinct = 1024, 128
    sigs = [bench.farm_signals(c) for c in range(distinct)]
    base = synth.make_capture_batch_torch([77_000 + c for c in range(distinct)], 1, table, sigs, "cuda").cpu().numpy()
    caps = base[np.arange(n_cap) % distinct]  # capture c is a copy of capture c % 128
    rec = nav_engine.search(caps.reshape(-1))
    assert rec.shape == (n_cap, 32)
    # (i) independence: identical captures give bitwise identical records wherever they sit in the batch
    for c in range(distinct, n_cap):
        assert rec[c].tobytes() == rec[c % distinct].tobytes()
    # (ii) batch == one-at-a-time
    for c in (0, 5, 77, 127):
        assert nav_engine.search(caps[c])[0].tobytes() == rec[c].tobytes()
    # (iii) the oracle on EVERY distinct capture
    m = Margins("cfg5, 128 distinct captures")
    ties = 0
    for c in range(distinct):
        orec, ogrid = oracle.search(caps[c], table, want_grid=True)
        ties += compare_records(rec[c], orec, ogrid, -20, 16.0, max_ties=1, margins=m)
    m.report()
    assert ties <= 4
    # (iv) every strong injected satellite is detected at its injected lag / Doppler bin
    for c in range(distinct):
        for sat, tau, f, cn0, _ in sigs[c]:
            if cn0 >= 45:
                r = rec[c][sat]
                assert r["snr"] >= 16 and abs(((r["lag"] - tau / 4.0 + 2046) % 4092) - 2046) <= 1
                assert r["dop"] == int(np.round(f / F.BIN_HZ))


def test_e1b_all_50_codes_against_reference_goldens(gpu_required):
    """The engine over all 50 Galileo E1-B codes against the UNMODIFIED search.cpp run over a 50-row table
    (oracle/_ref/libref_search_e1b50.so -> tests/golden/ref_e1b50.npz): code spectra of every PRN, and Correlate()'s
    answers on a capture synthesised from the reference's own chips.  Independent of the oracle and of every code
    table in this repository."""
    import os
    from conftest import GOLDEN
    g = np.load(os.path.join(GOLDEN, "ref_e1b50.npz"))
    table = S.e1b(range(1, 51))
    with F.AcqEngine(table) as eng:
        for k in range(50):
            c = eng.code_spectrum(k)
            scale = np.abs(g["spec_bins"][k]).max()
            assert np.abs(c[g["spec_idx"]] - g["spec_bins"][k]).max() / scale < 1e-5, k
            assert abs(np.abs(c).astype(np.float64).sum() / g["spec_abs_sum"][k] - 1) < 1e-5, k
        rec = eng.search(g["capture"])[0]
    thr = 16.0
    np.testing.assert_allclose(rec["snr"], g["snr"], rtol=RTOL)
    clear = np.abs(g["snr"] / thr - 1) > RTOL
    assert np.array_equal((rec["snr"] >= thr)[clear], (g["snr"] >= thr)[clear])
    det = g["snr"] >= thr * (1 + RTOL)
    assert np.array_equal(rec["dop"][det], g["dop"][det]) and np.array_equal(rec["lag"][det], g["lag"][det])
    assert np.array_equal(rec["dop"], g["dop"]) and np.array_equal(rec["lag"], g["lag"])  # no tie on this fixture
    print("e1b50: detected", int(det.sum()), "of 50; nearest to the threshold: snr", float(g["snr"][np.argmin(np.abs(g["snr"] - thr))]))


def test_e1b_noise_only_capture_near_the_threshold(cfg3_engine, oracle):
    """The E1B threshold (16, search.cpp:549) sits at the top of the noise distribution of a 16368-lag x 81-bin scan:
    this noise-only capture (seed found by tools/find_threshold_capture.py) has its strongest false peak within 3 % of
    16.  Engine and oracle must agree on which side every satellite falls, and the margin is printed."""
    table = scenarios.table("cfg3")
    kw = scenarios.params_kw("cfg3")
    cap = synth.make_capture(scenarios.E1B_NEAR_THRESHOLD_SEED, 1, table, [])
    rec, grid = cfg3_engine.search(cap, want_grid=True)
    orec, ogrid = oracle.search(cap, table, params=oracle.default_params(**kw), want_grid=True)
    m = Margins("noise-only E1B capture near the threshold")
    compare_records(rec[0], orec, ogrid, kw["dop_lo"], 16.0, ggrid=grid[0], max_ties=1, margins=m)
    m.report()
    top = float(orec["snr"].max())
    assert abs(top / 16.0 - 1) < 0.03, top
    assert np.array_equal(rec[0]["snr"] >= 16.0, orec["snr"] >= 16.0)


def test_farm_classes_with_the_cuda_engine(nav_engine, cfg4_engine):
    """farm.CaptureFarm / farm.SatFarm (the plumbing bench.py's multi-GPU lines run through) on one GPU with the CUDA
    engine: resident and end-to-end paths give the records of a plain acq_search, bitwise.  (World size 2 with uneven
    shards is covered under gloo on CPU; NCCL runs are bench.py --gpus N.)"""
    import torch
    from flydog_sdr_gps_b200 import farm
    table = S.navstar()
    caps = np.stack([synth.make_capture(300 + c, 1, table, scenarios.signals("cfg5", c)) for c in range(5)])
    want = nav_engine.search(caps.reshape(-1))
    st = torch.cuda.Stream()
    with torch.cuda.stream(st):
        f = farm.CaptureFarm(nav_engine, 5, 8192, 32)
        f.load(caps)
        got = f.search().copy()
        f.search_resident()
        st.synchronize()
        res = f.d_all.cpu().numpy().view(F.RECORD_DTYPE).reshape(5, 32)
    assert got.tobytes() == want.tobytes() and res.tobytes() == want.tobytes()
    assert (f.h2d_bytes, f.d2h_bytes) == (5 * 8192, 5 * 32 * 24)
    t4 = scenarios.table("cfg4")
    cap = synth.make_capture(41, 1, t4, scenarios.signals("cfg4", 1))
    with torch.cuda.stream(st):
        sf = farm.SatFarm(cfg4_engine, len(t4), 8192)
        sf.load(cap)
        rec = sf.search().copy()
    assert rec.tobytes() == cfg4_engine.search(cap)[0].tobytes()


def test_lag_and_doppler_sweep(nav_engine):
    """Round trip: inject one strong satellite at many (tau, Doppler); the record returns them."""
    table = S.navstar()
    rng = np.random.default_rng(8)
    caps, want = [], []
    for k in range(24):
        sat = int(rng.integers(0, 32))
        tau = int(rng.integers(0, 4092)) * 4
        dop = int(rng.integers(-20, 21))
        caps.append(synth.make_capture(100 + k, 1, table, [(sat, tau, dop * F.BIN_HZ, 50, float(rng.uniform(0, 6)))]))
        want.append((sat, tau // 4, dop))
    rec = nav_engine.search(np.concatenate(caps))
    for k, (sat, lag, dop) in enumerate(want):
        r = rec[k][sat]
        assert (r["lag"], r["dop"]) == (lag, dop) and r["snr"] > 50


def test_wrap_modes(gpu_required, oracle):
    """ACQ_WRAP_REFERENCE reproduces the compiled reference's row overrun; ACQ_WRAP_CIRCULAR the intended wrap."""
    table = S.reference_table()
    cap = synth.make_capture(77, 1, table, [(3, 777, -4000.0, 47, 0.1), (58, 40000, -2000.0, 47, 0.2)])
    sel = np.array([3, 31, 35, 36, 58], np.int32)
    for mode in (F.WRAP_REFERENCE, F.WRAP_CIRCULAR):
        with F.AcqEngine(table, F.default_params(wrap_mode=mode)) as eng:
            rec, grid = eng.search(cap, sel=sel, want_grid=True)
        orec, ogrid = oracle.search(cap, table, sel=sel, params=oracle.default_params(wrap_mode=mode), want_grid=True)
        compare_records(rec[0], orec, ogrid, -20, 16.0, ggrid=grid[0])


def test_selection_order_repeats_and_qzss(ref_engine, oracle):
    table = S.reference_table()
    cap = synth.make_capture(55, 1, table, [(33, 1234, 500.0, 48, 0.3), (2, 4444, -1000.0, 48, 0.3), (40, 50000, 0.0, 48, 1.0)])
    sel = np.array([40, 2, 33, 2, 58, 0], np.int32)  # mixed constellations, a repeat, arbitrary order
    rec = ref_engine.search(cap, sel=sel)[0]
    assert np.array_equal(rec["sat"], sel)
    orec, ogrid = oracle.search(cap, table, sel=sel, want_grid=True)
    compare_records(rec, orec, ogrid, -20, 16.0)
    assert rec[1].tobytes() == rec[3].tobytes()
    one = ref_engine.search(cap, sel=np.array([33], np.int32))[0]
    assert one[0].tobytes() == rec[2].tobytes()


def test_sbas_rows_are_zero_like_the_reference(gpu_required, oracle):
    """An SBAS row gets no replica (search.cpp:244): zero spectrum, record {lag 0, dop 0, snr 0}, and the row before it
    reads zeros at negative Doppler in the reference's wrap mode.  Engine against the oracle, whole per-Doppler table."""
    nav = S.navstar()
    table = nav[:3] + [(120, 145, 0o1106, S.SBAS)] + nav[3:6]
    cap = synth.make_capture(5, 1, nav, scenarios.signals("cfg1", 5))
    with F.AcqEngine(table) as eng:
        assert not eng.code_spectrum(3).any()
        rec, grid = eng.search(cap, want_grid=True)
    orec, ogrid = oracle.search(cap, table, want_grid=True)
    # reference wrap: the zero row reads the next row's first bins at negative Doppler (search.cpp:471): cells at
    # dop >= 0 are 0/0 -> NaN in both, the others small and equal to the oracle's
    assert np.array_equal(grid[0][3]["peak"], ogrid[3]["peak"]) or np.allclose(grid[0][3]["peak"], ogrid[3]["peak"], rtol=RTOL)
    assert (grid[0][3]["peak"][20:] == 0).all() and rec[0][3]["snr"] < 8
    assert (rec[0][3]["dop"], rec[0][3]["lag"]) == (orec[3]["dop"], orec[3]["lag"])
    keep = np.array([0, 1, 2, 4, 5, 6])
    compare_records(rec[0][keep], orec[keep], ogrid[keep], -20, 16.0, ggrid=grid[0][keep], max_ties=1)
    with F.AcqEngine(table, F.default_params(wrap_mode=F.WRAP_CIRCULAR)) as eng:
        r = eng.search(cap)[0][3]
    assert (r["sat"], r["lag"], r["dop"], r["peak"], r["noise"], r["snr"]) == (3, 0, 0, 0, 0, 0)


def test_degenerate_captures(nav_engine, oracle):
    """All-zero and all-one bit captures (a dead front end) follow the reference arithmetic too."""
    table = S.navstar()
    for fill in (0x00, 0xFF, 0xAA):
        cap = np.full(8192, fill, np.uint8)
        rec, grid = nav_engine.search(cap, sel=np.arange(4, dtype=np.int32), want_grid=True)
        orec, ogrid = oracle.search(cap, table, sel=np.arange(4), want_grid=True)
        ok = np.isfinite(ogrid["snr"])
        assert np.array_equal(np.isfinite(grid[0]["snr"]), ok)
        if ok.all():
            compare_records(rec[0], orec, ogrid, -20, 16.0, max_ties=4)


def test_asymmetric_doppler_range_and_single_bin(gpu_required, oracle):
    table = S.navstar()
    cap = synth.make_capture(66, 1, table, [(9, 2000, 3 * F.BIN_HZ, 48, 0.3)])
    for lo, hi in ((-3, 7), (3, 3), (-33, -30)):
        with F.AcqEngine(table, F.default_params(dop_lo=lo, dop_hi=hi)) as eng:
            rec, grid = eng.search(cap, sel=np.array([9, 10], np.int32), want_grid=True)
        orec, ogrid = oracle.search(cap, table, sel=[9, 10], params=oracle.default_params(dop_lo=lo, dop_hi=hi), want_grid=True)
        compare_records(rec[0], orec, ogrid, lo, 16.0, ggrid=grid[0], max_ties=1)


def test_async_submit_poll_wait(nav_engine):
    table = S.navstar()
    cap = synth.make_capture(3, 1, table, scenarios.signals("cfg1", 3))
    sync = nav_engine.search(cap)
    out = np.zeros(32, F.RECORD_DTYPE)
    nav_engine.submit(cap, out)
    with pytest.raises(F.AcqError):  # a second call while one is pending is refused, not queued silently
        nav_engine.search(cap)
    while not nav_engine.poll():
        pass
    nav_engine.wait()
    assert out.tobytes() == sync[0].tobytes()


def test_device_resident_api_on_torch_stream(nav_engine):
    import torch
    table = S.navstar()
    caps = np.concatenate([synth.make_capture(s, 1, table, scenarios.signals("cfg1", s)) for s in (1, 2, 3, 4)])
    host = nav_engine.search(caps)
    d_in = torch.from_numpy(caps).cuda()
    d_out = torch.zeros(4 * 32 * 24, dtype=torch.uint8, device="cuda")
    st = torch.cuda.Stream()
    with torch.cuda.stream(st):
        nav_engine.search_device(d_in.data_ptr(), d_out.data_ptr(), 4, stream_ptr=st.cuda_stream)
    st.synchronize()
    got = d_out.cpu().numpy().view(F.RECORD_DTYPE).reshape(4, 32)
    assert got.tobytes() == host.tobytes()
    n0 = nav_engine.launch_count
    nav_engine.search_device(d_in.data_ptr(), d_out.data_ptr(), 4)
    torch.cuda.synchronize()
    assert nav_engine.launch_count - n0 == 4  # front end, forward FFT, search, best-Doppler pick (k_pick_small)
    # interleaving: a device-path search on a torch stream, then the host path, then another stream, with a selection
    # change in between -- the engine orders them on its shared scratch (records bitwise equal each time)
    st2 = torch.cuda.Stream()
    sel = np.array([3, 9, 17, 30, 5], np.int32)
    host_sel = nav_engine.search(caps, sel=sel)
    d_out2 = torch.zeros(4 * 5 * 24, dtype=torch.uint8, device="cuda")
    for _ in range(3):
        nav_engine.search_device(d_in.data_ptr(), d_out.data_ptr(), 4, stream_ptr=st.cuda_stream)
        nav_engine.search_device(d_in.data_ptr(), d_out2.data_ptr(), 4, sel=sel, stream_ptr=st2.cuda_stream)
        assert nav_engine.search(caps).tobytes() == host.tobytes()
        torch.cuda.synchronize()
        assert d_out.cpu().numpy().tobytes() == host.tobytes()
        assert d_out2.cpu().numpy().tobytes() == host_sel.tobytes()
    # large batch: more than 256 rows, so the pick is k_best_dop behind the drained search and the records come back by a copy
    big = np.concatenate([caps] * 3)
    n0 = nav_engine.launch_count
    rec_big = nav_engine.search(big)
    assert nav_engine.launch_count - n0 == 4
    assert rec_big.tobytes() == (host.tobytes() * 3)


def test_engine_lifetime_leaves_no_device_memory_behind(gpu_required):
    """acq_create / searches through every host path / acq_destroy, thirty times: device memory returns to where it was
    (scratch, mapped staging buffers, events and streams are all owned by the handle)."""
    import torch
    table = S.reference_table()
    cap = synth.make_capture(11, 1, table, [(2, 4000, 4 * F.BIN_HZ, 48, 1.0)])
    sel = np.array([2, 40], np.int32)

    def cycle():
        with F.AcqEngine(table) as eng:
            r = eng.search(cap, sel=sel)                       # polled host path, tagged records
            eng.search(np.concatenate([cap] * 200), sel=sel)   # 400 rows: device records, copy, k_best_dop
            out = np.zeros((1, 2), F.RECORD_DTYPE)
            eng.submit(cap, out, sel=sel)
            eng.wait()
            assert out.tobytes() == r.tobytes()
            eng.refine(out)
    cycle()
    torch.cuda.synchronize()
    free0 = torch.cuda.mem_get_info()[0]
    for _ in range(30):
        cycle()
    torch.cuda.synchronize()
    assert free0 - torch.cuda.mem_get_info()[0] < (32 << 20)


def test_error_paths(nav_engine):
    L = _lib.load()
    cap = np.zeros(8192, np.uint8)
    with pytest.raises(F.AcqError) as ei:
        nav_engine.search(cap, sel=np.array([32], np.int32))
    assert ei.value.code == -1
    with pytest.raises(ValueError):
        nav_engine.search(np.zeros(100, np.uint8))
    out = np.zeros(32, F.RECORD_DTYPE)
    assert L.acq_search(nav_engine._h, None, 1, None, 0, out.ctypes.data) == -1
    assert L.acq_search(nav_engine._h, cap.ctypes.data, 0, None, 0, out.ctypes.data) == -1
    with pytest.raises(F.AcqError) as ei:
        F.AcqEngine(S.e1b([1, 2]), F.default_params(k_noncoh=300))
    assert ei.value.code == -1
    with pytest.raises(F.AcqError):
        F.AcqEngine(S.navstar(), F.default_params(dop_lo=5, dop_hi=-5))
    with pytest.raises(F.AcqError):
        F.AcqEngine([(1, 0, 6, 0)])
    # the engine is still usable after errors
    assert nav_engine.search(cap).shape == (1, 32)


def test_dropin_search_task_matches_literal_reference(gpu_required, golden_search):
    """The host shim replays the reference's SearchTask loop (search.cpp:512-604) against a mock receiver:
    same ChanReset / GPSstat / ChanStart calls, same order, same integer arguments as the unmodified
    reference produced on these captures (tests/golden/ref_search_task_events.npz)."""
    import os
    from conftest import GOLDEN
    from flydog_sdr_gps_b200 import dropin
    want = np.load(os.path.join(GOLDEN, "ref_search_task_events.npz"))["events"]
    rx = dropin.MockReceiver(golden_search["captures"], free_chans=12)
    d = dropin.Dropin(S.reference_table(), rx)
    started = d.search_pass(dropin.LITERAL) + d.search_pass(dropin.LITERAL)
    got = rx.events
    assert started == int((want["kind"] == 2).sum()) == 12
    assert len(got) == len(want)
    for g, w in zip(got, want):
        if w["kind"] == 1:
            assert g == ("chan_reset", w["a"], w["b"], w["c"])
        elif w["kind"] == 2:   # ChanStart(ch, sat, t_sample, lo_shift, ca_shift, (int) snr)
            assert g[:5] == ("chan_start", w["a"], w["b"], w["c"], w["d"])
            assert abs(g[5] - w["e"]) <= 1 and abs(g[5] - w["e"]) <= RTOL * w["e"] + 1
        elif w["kind"] == 3:   # GPSstat(STAT_SAT, snr, ch, sat, weak)
            assert g[0] == "stat_sat" and g[1:3] == (w["a"], w["b"])
            if abs(w["x"] / 16.0 - 1) > RTOL:
                assert g[3] == w["c"]
            assert abs(g[4] - w["x"]) <= RTOL * max(w["x"], 1e-9)
        elif w["kind"] == 4:   # GPSstat(STAT_DOP, ch, (int)(lo_shift*BIN_SIZE), ca_shift)
            assert g == ("stat_dop", w["a"], w["b"], w["c"])
    # SearchEnable re-arms a tracked satellite
    busy = [s for s in range(59) if d.is_busy(s)]
    assert len(busy) == 12
    d.enable(busy[0])
    assert not d.is_busy(busy[0])
    d.close()


def test_dropin_batch_mode_and_gsig(gpu_required, golden_search):
    """Capture-reuse mode (one capture, all idle sats in one GPU call) starts the same satellites the
    per-satellite search finds on that capture; -gsig raises the L1 threshold like SearchParams."""
    from flydog_sdr_gps_b200 import dropin
    cap = golden_search["captures"][0]
    rx = dropin.MockReceiver(cap, free_chans=12)
    d = dropin.Dropin(S.reference_table(), rx)
    n = d.search_pass(dropin.BATCH)
    started = sorted(e[2] for e in rx.events if e[0] == "chan_start")
    want = sorted(np.nonzero(golden_search["snr"][0] >= 16 * (1 + RTOL))[0].tolist())
    assert n == len(started) and set(want) <= set(started) and len(started) <= len(want) + 2
    for e in rx.events:
        if e[0] == "chan_start":
            assert e[3] == golden_search["dop"][0][e[2]] and e[4] == 4 * golden_search["lag"][0][e[2]]
    assert rx.samples == 1
    d.close()
    rx2 = dropin.MockReceiver(cap, free_chans=12)
    d2 = dropin.Dropin(S.reference_table(), rx2)
    d2.params("-gsig", "60")
    d2.set_acq(1, 0, 0)
    d2.search_pass(dropin.LITERAL)
    started2 = sorted(e[2] for e in rx2.events if e[0] == "chan_start")
    assert started2 == sorted(np.nonzero(golden_search["snr"][0][:32] >= 60)[0].tolist())
    assert all(e[1] < 32 for e in rx2.events if e[0] == "chan_reset")
    d2.close()


def test_e1b_cluster_kernel_equals_single_cta_kernel(gpu_required, oracle):
    """The cluster/DSMEM form of the E1B search (four CTAs per tile) against the one-CTA-per-tile form on the same
    capture: same sub-FFTs and combine, so peaks and lags are bitwise equal; only the order of the noise sum
    differs.  Both against the oracle."""
    table = scenarios.table("cfg3")[:12]
    kw = scenarios.params_kw("cfg3")
    cap = synth.make_capture(33, 1, table, [(1, 30000, -6 * F.BIN_HZ, 47, 0.4), (7, 1000, 31 * F.BIN_HZ, 46, 1.4),
                                            (11, 65000, 0.0, 45, 2.4)])
    out = {}
    for kind in ("cta", "cluster"):   # variant libraries that force one form (the product picks by tile count)
        with F.AcqEngine(table, F.default_params(**kw), variant="e1b_" + kind) as eng:
            out[kind] = eng.search(cap, want_grid=True)
    (ra, ga), (rb, gb) = out["cta"], out["cluster"]
    assert np.array_equal(ga["peak"], gb["peak"]) and np.array_equal(ga["lag"], gb["lag"])
    np.testing.assert_allclose(ga["noise"], gb["noise"], rtol=2e-6)
    assert np.array_equal(ra["lag"], rb["lag"]) and np.array_equal(ra["dop"], rb["dop"])
    orec, ogrid = oracle.search(cap, table, params=oracle.default_params(**kw), want_grid=True)
    compare_records(rb[0], orec, ogrid, kw["dop_lo"], 16.0, ggrid=gb[0], max_ties=1)
    assert {int(r["sat"]) for r in rb[0] if r["snr"] >= 16} >= {1, 7, 11}


def test_e1b_tma_staged_kernel_equals_ldg_kernel(gpu_required, oracle):
    """The operand-staging E1B kernel (TMA bulk copies one sub-FFT ahead, deferred peak merge) against the earlier
    load-from-L2 form: the arithmetic is the same instruction for instruction, so the whole grid is bitwise equal.
    More tiles than resident CTAs, so the deferred merge and the cross-tile prefetch are exercised."""
    table = scenarios.table("cfg3")[:9]
    kw = scenarios.params_kw("cfg3")
    cap = synth.make_capture(37, 1, table, [(0, 12345, 17 * F.BIN_HZ, 47, 0.4), (8, 64000, -39 * F.BIN_HZ, 46, 1.4)])
    out = {}
    for kind, variant in (("tma", "e1b_cta"), ("ldg", "e1b_ldg")):
        with F.AcqEngine(table, F.default_params(**kw), variant=variant) as eng:
            out[kind] = eng.search(cap, want_grid=True)
    (ra, ga), (rb, gb) = out["tma"], out["ldg"]
    for f in ("peak", "lag", "noise", "snr"):
        assert np.array_equal(ga[f], gb[f]), f
    assert np.array_equal(ra, rb)
    orec, ogrid = oracle.search(cap, table, params=oracle.default_params(**kw), want_grid=True)
    compare_records(ra[0], orec, ogrid, kw["dop_lo"], 16.0, ggrid=ga[0], max_ties=1)
    assert {int(r["sat"]) for r in ra[0] if r["snr"] >= 16} >= {0, 8}


def test_e1b_noncoherent_blocks(gpu_required, oracle):
    """Galileo E1B with K = 4 non-coherent blocks and half-bin Doppler (cluster kernel, block powers summed in
    registers per lag quarter) against the oracle's extension of search.cpp."""
    table = scenarios.table("cfg3")[:10]
    kw = dict(dop_lo=-12, dop_hi=12, half_bin=1, k_noncoh=4, thr_e1b=8.0)
    cap = synth.make_capture(35, 4, table, [(2, 20000, 3.5 * F.BIN_HZ, 40, 0.3), (6, 61000, -2 * F.BIN_HZ, 39, 1.1)])
    with F.AcqEngine(table, F.default_params(**kw)) as eng:
        rec, grid = eng.search(cap, want_grid=True)
    orec, ogrid = oracle.search(cap, table, params=oracle.default_params(**kw), want_grid=True)
    compare_records(rec[0], orec, ogrid, kw["dop_lo"], kw["thr_e1b"], ggrid=grid[0], max_ties=1)
    assert {int(r["sat"]) for r in rec[0] if r["snr"] >= kw["thr_e1b"]} >= {2, 6}


def test_e1b_one_cta_multi_kernel_equals_cluster_kernel(gpu_required, oracle):
    """k_search_e1b_multi (K > 1 on one CTA per tile: block powers split between tensor memory and a shared-memory
    array, code operand straight from L2) against the cluster/DSMEM form with K > 1 (variant library e1b_cluster): same
    sub-FFTs, combine and block order, so peaks and lags are bitwise equal; only the order of the noise sum differs.
    More tiles than resident CTAs; both against the oracle."""
    table = scenarios.table("cfg3")[:16]
    kw = dict(dop_lo=-20, dop_hi=20, k_noncoh=3, thr_e1b=7.0)
    cap = synth.make_capture(39, 3, table, [(1, 30000, -6 * F.BIN_HZ, 42, 0.4), (7, 1000, 17 * F.BIN_HZ, 41, 1.4),
                                            (12, 65000, 0.0, 40, 2.4)])
    out = {}
    for kind, variant in (("cta", None), ("cluster", "e1b_cluster")):
        with F.AcqEngine(table, F.default_params(**kw), variant=variant) as eng:
            out[kind] = eng.search(cap, want_grid=True)
    (ra, ga), (rb, gb) = out["cta"], out["cluster"]
    assert np.array_equal(ga["peak"], gb["peak"]) and np.array_equal(ga["lag"], gb["lag"])
    np.testing.assert_allclose(ga["noise"], gb["noise"], rtol=2e-6)
    assert np.array_equal(ra["lag"], rb["lag"]) and np.array_equal(ra["dop"], rb["dop"])
    orec, ogrid = oracle.search(cap, table, params=oracle.default_params(**kw), want_grid=True)
    compare_records(ra[0], orec, ogrid, kw["dop_lo"], kw["thr_e1b"], ggrid=ga[0], max_ties=1)
    assert {int(r["sat"]) for r in ra[0] if r["snr"] >= kw["thr_e1b"]} >= {1, 7, 12}


def test_dropin_with_capture_file_source(gpu_required, golden_search, tmp_path):
    """GPS_SAMPLES_FROM_FILE path (gps/search.cpp:361-380): the shim's capture callback fed from a raw capture
    file gives the same detections as the golden per-capture answers, and the file's end stops the pass."""
    from flydog_sdr_gps_b200 import capture, dropin
    caps = golden_search["captures"]
    path = tmp_path / "captures.if.4092.dat"
    path.write_bytes(np.ascontiguousarray(caps[:2]).tobytes())
    src = capture.CaptureFile(path)

    class FileReceiver(dropin.MockReceiver):
        def capture(self, _u, dst):
            blk = src.next()
            if blk is None:
                return 1
            C.memmove(dst, blk.ctypes.data, 8192)
            self.samples += 1
            return 0

    rx = FileReceiver(caps[0], free_chans=12)
    d = dropin.Dropin(S.reference_table(), rx)
    for k in range(2):   # batch mode: one capture from the file per pass
        rx.events.clear()
        rx.free, rx.next_ch = 12, 0
        for s in range(59):
            d.enable(s)
        d.search_pass(dropin.BATCH)
        started = {e[2]: e for e in rx.events if e[0] == "chan_start"}
        strong = np.nonzero(golden_search["snr"][k] >= 16 * (1 + RTOL))[0]
        assert set(strong.tolist()) <= set(started)
        for sat in strong:
            assert started[sat][3] == golden_search["dop"][k][sat] and started[sat][4] == 4 * golden_search["lag"][k][sat]
    with pytest.raises(RuntimeError):   # end of file: the capture callback fails, the pass reports it
        d.search_pass(dropin.BATCH)
    assert rx.samples == 2
    d.close()
    src.close()


# ---------------------------------------------------------------- acquisition refinement (SURVEY 8(f) rank 4)
def _compare_fine(gfine, ofine, rec):
    g, o, r = np.asarray(gfine).reshape(-1), np.asarray(ofine).reshape(-1), np.asarray(rec).reshape(-1)
    assert np.allclose(g["peak"], o["peak"], rtol=RTOL)
    assert np.allclose(g["peak"], r["peak"], rtol=RTOL)  # the direct sum reproduces the FFT search's peak cell
    # interpolation offsets: 2e-3 of a bin / of a /4 sample (fp32 sums of 16384 terms against the oracle's doubles)
    assert np.abs(g["dop_hz"] - o["dop_hz"]).max() < 2e-3 * F.BIN_HZ, np.abs(g["dop_hz"] - o["dop_hz"]).max()
    assert np.abs(g["code_fs"] - o["code_fs"]).max() < 8e-3, np.abs(g["code_fs"] - o["code_fs"]).max()
    away = np.abs((o["code_fs"] % 1.0) - 0.5) > 0.02  # rounding to whole FS samples, away from the .5 boundary
    assert np.array_equal(g["ca_shift"][away], o["ca_shift"][away])


def test_refine_matches_oracle_and_injected_values(ref_engine, oracle):
    table = S.reference_table()
    sig = [(2, 4001, 3.3 * F.BIN_HZ, 50, 1.0), (10, 12346, -7.45 * F.BIN_HZ, 48, 2.0), (44, 30003, -6.2 * F.BIN_HZ, 50, 0.4)]
    cap = synth.make_capture(77, 1, table, sig)
    sel = np.array([2, 10, 44, 20, 58], np.int32)
    rec = ref_engine.search(cap, sel=sel)
    fine = ref_engine.refine(rec)
    assert fine.shape == rec.shape
    _compare_fine(fine, oracle.refine(cap, table, rec[0]), rec)
    for i, (sat, tau, fd, _, _) in enumerate(sig):
        period = 4 * (F.LAGS_E1B if table[sat][3] == S.E1B else F.LAGS_L1)
        err = (float(fine["code_fs"][0, i]) - tau) % period
        err = err - period if err > period / 2 else err
        assert abs(fine["dop_hz"][0, i] - fd) < 0.25 * F.BIN_HZ and abs(err) < 2.0


def test_refine_half_bins_noncoherent_and_batches(gpu_required, oracle):
    table = S.navstar()
    kw = dict(k_noncoh=4, half_bin=1, dop_lo=-20, dop_hi=20)
    caps = [synth.make_capture(78 + c, 4, table, [(7, 8002 + c, (4.5 - c) * F.BIN_HZ, 46, 0.5), (12, 100, -3.1 * F.BIN_HZ, 46, 0.1)])
            for c in range(3)]
    sel = np.array([7, 12, 30], np.int32)
    with F.AcqEngine(table, F.default_params(**kw)) as eng:
        rec = eng.search(np.concatenate(caps), sel=sel)
        fine = eng.refine(rec)
        for c in range(3):
            _compare_fine(fine[c], oracle.refine(caps[c], table, rec[c], params=oracle.default_params(**kw)), rec[c])
        assert abs(fine["dop_hz"][0, 0] - 4.5 * F.BIN_HZ) < 0.25 * F.BIN_HZ
        # refining again gives the same bytes (no state is consumed)
        assert eng.refine(rec).tobytes() == fine.tobytes()


def test_refine_error_paths(gpu_required):
    table = S.navstar()
    cap = synth.make_capture(5, 1, table, [(3, 400, 0.0, 50, 0.0)])
    with F.AcqEngine(table) as eng:
        with pytest.raises(F.AcqError):  # nothing searched yet
            eng.refine(np.zeros(32, F.RECORD_DTYPE))
        rec = eng.search(cap)
        with pytest.raises(F.AcqError):  # wrong count
            eng.refine(rec[0, :5])
        bad = rec.copy()
        bad["sat"][0, 0] = 7             # not the satellite of that slot
        with pytest.raises(F.AcqError):
            eng.refine(bad)
        bad = rec.copy()
        bad["lag"][0, 1] = 5000          # outside the 1 ms window
        with pytest.raises(F.AcqError):
            eng.refine(bad)
        assert eng.refine(rec).shape == rec.shape


def test_dropin_refined_handoff(gpu_required, golden_search):
    """With acq_dropin_set_refine the shim hands ChanStart a ca_shift at FS-sample resolution (within one /4 sample of
    lag * DECIM) and the bin nearest to the interpolated Doppler (at most one bin from the search's); the started
    set, call order and units are those of the unrefined pass.  Literal and batch mode agree."""
    from flydog_sdr_gps_b200 import dropin
    cap = golden_search["captures"][0]
    table = S.reference_table()
    runs = {}
    for mode in (dropin.LITERAL, dropin.BATCH):
        for refine in (0, 1):
            rx = dropin.MockReceiver(cap, free_chans=59)
            d = dropin.Dropin(table, rx)
            d.set_refine(refine)
            d.search_pass(mode)
            runs[mode, refine] = {e[2]: (e[3], e[4]) for e in rx.events if e[0] == "chan_start"}
            d.close()
    for mode in (dropin.LITERAL, dropin.BATCH):
        plain, fine = runs[mode, 0], runs[mode, 1]
        assert plain.keys() == fine.keys() and len(plain) >= 5
        for sat in plain:
            period = 4 * (F.LAGS_E1B if table[sat][3] == S.E1B else F.LAGS_L1)
            dca = (fine[sat][1] - plain[sat][1] + period // 2) % period - period // 2
            assert abs(dca) <= 4 and 0 <= fine[sat][1] < period
            assert abs(fine[sat][0] - plain[sat][0]) <= 1
    assert runs[dropin.LITERAL, 1] == runs[dropin.BATCH, 1]


def test_sign_magnitude_captures(gpu_required, oracle):
    """2-bit sign/magnitude capture format (acq_params.sample_bits = 2, an extension: the MAX2769 produces I_mag,
    the reference's FPGA drops it).  Front end bit-exact against the oracle's definition, search parity for K = 1
    and for half-bin K = 3 sums, and an all-zero magnitude plane equals the 1-bit engine byte for byte."""
    table = S.navstar()
    sig = scenarios.signals("cfg1", 2)
    c1 = synth.make_capture(2, 1, table, sig)
    c2 = synth.make_capture(2, 1, table, sig, sample_bits=2)
    with F.AcqEngine(table) as e1, F.AcqEngine(table, F.default_params(sample_bits=2)) as e2:
        assert e2.block_bytes == 16384 and e1.block_bytes == 8192
        x2, D = e2.capture_spectrum(c2)
        assert np.array_equal(x2, oracle.capture_baseband(c2, 0, 2))
        x2h, _ = e2.capture_spectrum(c2, 1)
        assert np.array_equal(x2h, oracle.capture_baseband(c2, 1, 2))
        rec, grid = e2.search(c2, want_grid=True)
        orec, ogrid = oracle.search(c2, table, params=oracle.default_params(sample_bits=2), want_grid=True)
        compare_records(rec[0], orec, ogrid, -20, 16.0, ggrid=grid[0])
        one = e1.search(c1)
        strong = one[0]["snr"] >= 30
        assert strong.sum() >= 3 and (rec[0]["snr"][strong] > one[0]["snr"][strong]).all()  # less quantisation loss
        assert np.array_equal(rec[0]["lag"][strong], one[0]["lag"][strong])
        z = np.concatenate([c1, np.zeros(8192, np.uint8)])
        assert e2.search(z).tobytes() == one.tobytes()
        # two captures in one call: capture stride is 16384 bytes
        both = e2.search(np.concatenate([z, c2]))
        assert both[0].tobytes() == one[0].tobytes() and both[1].tobytes() == rec[0].tobytes()
        with pytest.raises(ValueError):
            e2.search(c1)  # a 1-bit capture is half a block in this engine's format
    kw = dict(dop_lo=-12, dop_hi=12, half_bin=1, k_noncoh=3, thr_l1=8.0, sample_bits=2)
    sig = [(4, 5000, 2.5 * F.BIN_HZ, 40, 0.2), (20, 16000, -1.0 * F.BIN_HZ, 41, 1.2)]
    cap = synth.make_capture(12, 3, table, sig, sample_bits=2)
    sel = np.array([4, 20, 7], np.int32)
    with F.AcqEngine(table, F.default_params(**kw)) as eng:
        rec, grid = eng.search(cap, sel=sel, want_grid=True)
        fine = eng.refine(rec)
    orec, ogrid = oracle.search(cap, table, sel=sel, params=oracle.default_params(**kw), want_grid=True)
    compare_records(rec[0], orec, ogrid, kw["dop_lo"], kw["thr_l1"], ggrid=grid[0], max_ties=1)
    assert rec[0]["dop"][0] == 5 and rec[0]["dop"][1] == -2
    assert np.allclose(fine[0]["peak"], rec[0]["peak"], rtol=1e-4)
    with pytest.raises(F.AcqError):
        F.AcqEngine(table, F.default_params(sample_bits=3))


def test_code_doppler_compensation(gpu_required, oracle):
    """acq_params.code_doppler: shifted copies of the capture spectra, selected per (block, Doppler index) in the
    search kernels and in the refinement -- against the oracle's per-block lag shift on a capture whose codes are
    stretched by their carrier offsets.  C/A (TMA-staged and LDG forms), half-bins, and E1B non-coherent sums."""
    table = S.navstar()
    BIN = F.BIN_HZ
    K = 12
    kw = dict(dop_lo=-80, dop_hi=80, half_bin=1, k_noncoh=K, thr_l1=3.0, code_doppler=1)
    sig = [(4, 5000, 38.0 * BIN, 37, 0.2), (20, 16000, -37.5 * BIN, 37, 1.2), (9, 800, 1.0 * BIN, 37, 0.7)]
    cap = synth.make_capture(5, K, table, sig, code_doppler=True)
    sel = np.array([4, 20, 9, 11], np.int32)
    orec, ogrid = oracle.search(cap, table, sel=sel, params=oracle.default_params(**kw), want_grid=True)
    with F.AcqEngine(table, F.default_params(**kw)) as eng:
        rec, grid = eng.search(cap, sel=sel, want_grid=True)
        fine = eng.refine(rec)
        two = eng.search(np.concatenate([cap, cap]), sel=sel)       # capture stride with shifted copies
    compare_records(rec[0], orec, ogrid, kw["dop_lo"], kw["thr_l1"], ggrid=grid[0], max_ties=1)
    assert np.array_equal(rec[0]["dop"][:3], [76, -75, 2]) and np.array_equal(rec[0]["lag"][:3], [1250, 4000, 200])
    assert two[0].tobytes() == rec[0].tobytes() and two[1].tobytes() == rec[0].tobytes()
    ofine = oracle.refine(cap, table, orec, params=oracle.default_params(**kw))
    assert np.allclose(fine[0]["peak"], rec[0]["peak"], rtol=1e-4)
    assert np.abs(fine[0]["dop_hz"][:3] - ofine["dop_hz"][:3]).max() < 2e-3 * BIN
    kw0 = dict(kw, code_doppler=0)
    with F.AcqEngine(table, F.default_params(**kw0)) as eng:
        plain = eng.search(cap, sel=sel)
    assert (rec[0]["snr"][:2] > 1.05 * plain[0]["snr"][:2]).all()    # the compensation recovers the smeared peaks
    assert rec[0][2].tobytes() == plain[0][2].tobytes()              # |h| = 2: no shift in any block
    # E1B, full bins, K = 6 (cluster kernel with block sums)
    gal = S.e1b([3, 11, 19])
    kwe = dict(dop_lo=-40, dop_hi=40, k_noncoh=6, thr_e1b=5.0, code_doppler=1)
    sige = [(1, 30000, -39.0 * BIN, 40, 0.4)]
    cape = synth.make_capture(8, 6, gal, sige, code_doppler=True)
    orec, ogrid = oracle.search(cape, gal, params=oracle.default_params(**kwe), want_grid=True)
    with F.AcqEngine(gal, F.default_params(**kwe)) as eng:
        rec, grid = eng.search(cape, want_grid=True)
    compare_records(rec[0], orec, ogrid, -40, 5.0, ggrid=grid[0], max_ties=1)
    assert rec[0]["dop"][1] == -39 and rec[0]["snr"][1] >= 5.0


def test_capture_resident_kernel_equals_cta_kernel(gpu_required, oracle):
    """k_search_l1_cr (the K = 1 full-bin product kernel: two CTAs per SM, the capture residue parked in tensor memory,
    chunks of 16 / 4 / 1 consecutive tiles claimed from a counter once a launch has six rounds of tiles, the static stride
    below) against k_search_l1<false> (two CTAs per SM striding over the tiles, both operands staged per sub-FFT; variant
    library l1_cta): the same arithmetic in the same order, so the whole per-Doppler table is bitwise equal.  Shapes: one
    capture, 40 captures (capture boundaries inside chunks), one capture 40 times (more tiles than resident CTAs; every
    copy's table equals the first's), 600 two-tile captures (several boundaries per chunk, alternating captures so that a
    residue left over from the neighbour would show), fewer tiles than SMs, a single tile."""
    table = S.navstar()
    cap = synth.make_capture(3, 1, table, scenarios.signals("cfg1", 3))
    cap2 = synth.make_capture(5, 1, table, scenarios.signals("cfg1", 5))
    cases = [({}, [cap], None), ({}, [cap, cap2] * 20, None), ({}, [cap] * 40, None),
             (dict(dop_lo=3, dop_hi=4), [cap, cap2] * 300, np.array([2], np.int32)),
             (dict(dop_lo=-3, dop_hi=1), [cap2], np.array([2], np.int32)),
             (dict(dop_lo=0, dop_hi=0), [cap], np.array([6], np.int32)),
             (dict(dop_lo=-20, dop_hi=20), [cap2, cap], np.array([2, 6, 10, 13, 18], np.int32))]
    for kw, caps, sel in cases:
        out = {}
        # product: k_search_l1_cr (claiming from six rounds of tiles)
        # cr: k_search_l1_cr (capture resident, chunks of tiles claimed) at every size -- the variant that always claims
        for kind, variant in (("product", None), ("cr", "dyn_tiles"), ("cta", "l1_cta")):
            with F.AcqEngine(table, F.default_params(**kw), variant=variant) as eng:
                out[kind] = eng.search(np.concatenate(caps), sel=sel, want_grid=True)
        rb, gb = out["cta"]
        for kind in ("product", "cr"):
            ra, ga = out[kind]
            for f in ("peak", "lag", "noise", "snr"):
                assert np.array_equal(ga[f], gb[f]), (kind, kw, len(caps), f)
            assert ra.tobytes() == rb.tobytes(), kind
        if all(c is caps[0] for c in caps):   # one capture repeated: every copy's table is the first's
            assert (out["product"][1][0] == out["product"][1][-1]).all()
    # half-bin K = 1 searches stay on k_search_l1<false> (odd and even half-bins read different capture spectra)
    with F.AcqEngine(table, F.default_params(half_bin=1, dop_lo=-9, dop_hi=9)) as eng:
        rec, grid = eng.search(cap, want_grid=True)
    orec, ogrid = oracle.search(cap, table, params=oracle.default_params(half_bin=1, dop_lo=-9, dop_hi=9), want_grid=True)
    compare_records(rec[0], orec, ogrid, -9, 16.0, ggrid=grid[0], max_ties=1)


def test_code_resident_multi_kernel_equals_twiddle_resident_kernel(gpu_required, oracle):
    """k_search_l1_multi (K > 1: the tile's code run parked in tensor memory after block 0, stage-B twiddles from a
    shared-memory table) against k_search_l1<true> (twiddles in tensor memory, code run staged for every block; variant
    library l1_multi_tw): the same arithmetic in the same order, so the whole per-Doppler table is bitwise equal --
    K = 20 half-bins (cfg2), K = 3 full bins over three captures with an asymmetric Doppler range, and K = 5 half-bins
    with code-Doppler copies."""
    table = S.navstar()
    cases = [(scenarios.params_kw("cfg2"), synth.make_capture(26, 20, table, scenarios.signals("cfg2", 6)), 1),
             (dict(dop_lo=-7, dop_hi=30, k_noncoh=3, thr_l1=8.0), synth.make_capture(27, 3, table, scenarios.signals("cfg1", 7)), 3),
             (dict(dop_lo=-60, dop_hi=60, half_bin=1, k_noncoh=5, thr_l1=5.0, code_doppler=1),
              synth.make_capture(4, 5, table, scenarios.signals("cfg2", 2), code_doppler=True), 1)]
    for kw, cap, reps in cases:
        out = {}
        # product: k_search_l1_multi; l1_multi_tw: k_search_l1<true>
        for kind, variant in (("code", None), ("tw", "l1_multi_tw")):
            with F.AcqEngine(table, F.default_params(**kw), variant=variant) as eng:
                out[kind] = eng.search(np.concatenate([cap] * reps), want_grid=True)
        (ra, ga), (rb, gb) = out["code"], out["tw"]
        for f in ("peak", "lag", "noise", "snr"):
            assert np.array_equal(ga[f], gb[f]), (kw, f)
        assert ra.tobytes() == rb.tobytes(), kw
        assert (ga[0] == ga[-1]).all()


@pytest.mark.parametrize("seed", range(12))
def test_randomized_parameter_space(gpu_required, oracle, seed):
    """Seeded sweep over the parameter space the C ABI accepts -- Doppler range (symmetric or not), half-bins,
    K blocks, wrap mode, capture format, code-Doppler compensation, mixed-constellation selections in random order --
    each case against the oracle on the same bytes, records and full per-Doppler tables."""
    rng = np.random.default_rng(9000 + seed)
    table = S.reference_table()
    half = int(rng.integers(0, 2))
    K = int(rng.choice([1, 1, 2, 3, 5]))
    span = int(rng.integers(2, 30)) * (2 if half else 1)
    lo = -int(rng.integers(0, span + 1))
    hi = lo + span
    bits = int(rng.choice([1, 2]))
    kw = dict(dop_lo=lo, dop_hi=hi, half_bin=half, k_noncoh=K, wrap_mode=int(rng.integers(0, 2)), sample_bits=bits,
              code_doppler=int(rng.integers(0, 2)), thr_l1=16.0 if K == 1 else 6.0, thr_e1b=16.0 if K == 1 else 6.0)
    sel = rng.choice(len(table), size=int(rng.integers(1, 7)), replace=False).astype(np.int32)
    step = F.BIN_HZ / (2 if half else 1)
    sig = []
    for s in sel[:3]:   # up to three of the searched satellites are present, inside the searched span
        period = 65472 if table[s][3] == S.E1B else 16368
        sig.append((int(s), int(rng.integers(0, period)), float(rng.uniform(lo, hi)) * step,
                    float(rng.uniform(44, 50)), float(rng.uniform(0, 6.28))))
    cap = synth.make_capture(500 + seed, K, table, sig, sample_bits=bits, code_doppler=bool(kw["code_doppler"]))
    with F.AcqEngine(table, F.default_params(**kw)) as eng:
        rec, grid = eng.search(cap, sel=sel, want_grid=True)
    orec, ogrid = oracle.search(cap, table, sel=sel, params=oracle.default_params(**kw), want_grid=True)
    thr = np.array([kw["thr_e1b"] if table[s][3] == S.E1B else kw["thr_l1"] for s in sel])
    for i in range(len(sel)):   # per-constellation thresholds: compare record by record
        compare_records(rec[0][i:i + 1], orec[i:i + 1], ogrid[i:i + 1], lo, float(thr[i]), ggrid=grid[0][i:i + 1], max_ties=1)
    assert np.array_equal(rec[0]["sat"], sel)


def test_capture_as_kernel_argument_equals_copied_capture(gpu_required):
    """acq_search of ONE 1-bit block hands the capture to the front end as a kernel argument (k_front_end_arg; no staging,
    no copy node); every other search copies it to the device first.  Same bits in, same front-end arithmetic: the records
    and the whole per-Doppler table are bytewise equal to the variant library that always copies (argin0), for a table
    with C/A and E1B rows, and a two-capture search (copied in both builds) still matches its single-capture halves."""
    table = scenarios.table("cfg4")
    kw = scenarios.params_kw("cfg4")
    caps = [synth.make_capture(s, 1, table, scenarios.signals("cfg4", s)) for s in (11, 12)]
    out = {}
    for kind, variant in (("arg", None), ("copy", "argin0")):
        with F.AcqEngine(table, F.default_params(**kw), variant=variant) as eng:
            out[kind] = [eng.search(c, want_grid=True) for c in caps] + [eng.search(np.concatenate(caps), want_grid=True)]
    for (ra, ga), (rb, gb) in zip(out["arg"], out["copy"]):
        assert ra.tobytes() == rb.tobytes()
        assert ga.tobytes() == gb.tobytes()
    both_r, both_g = out["arg"][2]
    for i in range(2):
        assert both_r[i].tobytes() == out["arg"][i][0][0].tobytes()
        assert both_g[i].tobytes() == out["arg"][i][1][0].tobytes()


def test_claimed_tiles_equal_static_stride(gpu_required):
    """The strided search kernels (k_search_l1<false>, k_search_l1_multi, k_search_e1b, k_search_e1b_multi) claim their tiles
    from a counter instead of striding by the grid size once a launch has six rounds of them (the two CTAs of an SM do not
    progress at the same rate).  Which CTA
    runs a tile cannot change its cell: records and the whole per-Doppler table are bytewise equal to the static stride
    (variant static_tiles), over repeated searches on one engine (the counter must come back to zero by itself), for
    searches of fewer tiles than CTAs, exactly one tile, and many rounds."""
    cases = [("cfg4", {}, None, 3), ("cfg4", {}, np.array([3, 40], np.int32), 2), ("cfg1", dict(dop_lo=2, dop_hi=2), np.array([5], np.int32), 2),
             ("cfg2", dict(dop_lo=-12, dop_hi=11), np.array([0, 9, 17], np.int32), 2), ("cfg3_k4", dict(dop_lo=-6, dop_hi=6), None, 2)]
    for cfg, over, sel, reps in cases:
        table = scenarios.table(cfg)
        kw = dict(scenarios.params_kw(cfg))
        kw.update(over)
        K = kw.get("k_noncoh", 1)
        caps = [synth.make_capture(70 + i, K, table, scenarios.signals(cfg, 70 + i)) for i in range(2)]
        out = {}
        # product: claims from six rounds of tiles up; dyn_tiles: always; static_tiles: never
        for kind, variant in (("product", None), ("claimed", "dyn_tiles"), ("static", "static_tiles")):
            with F.AcqEngine(table, F.default_params(**kw), variant=variant) as eng:
                out[kind] = [eng.search(caps[i % 2], sel=sel, want_grid=True) for i in range(reps)]
                out[kind].append(eng.search(np.concatenate(caps), sel=sel, want_grid=True))
        for kind in ("product", "claimed"):
            for (ra, ga), (rb, gb) in zip(out[kind], out["static"]):
                assert ra.tobytes() == rb.tobytes(), (kind, cfg, over)
                assert ga.tobytes() == gb.tobytes(), (kind, cfg, over)
