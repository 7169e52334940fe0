"""GPU suite (-m gpu) of the coherent search (acq_search_coherent) over its shape space, against the float64 reference
(tests/coherent_ref.py): a seeded sweep of M, groups, Doppler grids, capture formats, wraps, captures per call and
selections; searches of many tiles per persistent CTA; data-bit edges before every block of a group and mid-block; the
largest Doppler span; and a batch of more than 32 768 block rows (the launch split of k_coh_variants)."""
import numpy as np
import pytest

import flydog_sdr_gps_b200 as F
from flydog_sdr_gps_b200 import synth
from flydog_sdr_gps_b200 import sats as S

import search_ref
from coherent_ref import CoherentRef, grid_h
from search_ref import SNR_RTOL, Worst
from test_gpu_limits import SPLIT_CAPTURES, SPLIT_DISTINCT, SPLIT_K, SPLIT_PAST, SPLIT_STRADDLE, split_batch

pytestmark = pytest.mark.gpu
BIN = F.BIN_HZ
SBAS_ROW = 32


def _table():
    """32 Navstar rows, an SBAS row (no replica: a zero code row) and the 4 QZSS rows."""
    return S.navstar() + [(120, 145, 0o1106, S.SBAS)] + S.qzss()


def check_cells(g, ref, m_coh, hs=None, worst=None, what=""):
    """GPU cells g (at the Doppler indices hs, default the whole row) against the reference at search_ref's tolerances
    (search_ref.check_cells: peak, noise, snr, and the lag wherever the reference's power at the GPU's lag is not
    within PEAK_RTOL of its peak); the cells of a zero code row are 0 / 0 = NaN on both sides.  Returns the
    reference's (hs, snr)."""
    with np.errstate(invalid="ignore", divide="ignore"):
        cells = ref.cells(m_coh, hs=hs)
    hs, peak, noise, snr = cells[:4]
    assert g.size == hs.size
    search_ref.check_cells(g, cells, Worst() if worst is None else worst, what)
    zero = ~(noise > 0)
    assert (g["peak"][zero] == 0).all() and (g["noise"][zero] == 0).all() and np.isnan(g["snr"][zero]).all(), what
    return hs, snr


def check_record(r, g, hs, snr):
    """The record of a whole row: the cell of the best snr (lowest index on ties) wherever the reference's runner-up is
    not within SNR_RTOL of its best; a row whose snr never exceeds 0 keeps {dop 0, lag 0}."""
    s = np.where(np.isfinite(snr), snr, -np.inf)
    if not s.max() > 0:
        assert (r["dop"], r["lag"]) == (0, 0)
        return
    b = int(np.argmax(s))
    runner = np.sort(s)[-2] if s.size > 1 else -np.inf
    if runner < s[b] * (1 - SNR_RTOL):
        assert r["dop"] == hs[b] and r["lag"] == g["lag"][b] and r["peak"] == g["peak"][b], (r, hs[b])


# ---------------------------------------------------------------- seeded sweep
RANGE_KINDS = ["symmetric", "asymmetric", "positive", "negative", "single"]


def _sweep_case(seed):
    rng = np.random.default_rng(7100 + seed)
    if seed == 0:   # K = 255: 51 groups of M = 5, on a narrow range
        M, G = 5, 51
    else:
        M, G = int(rng.integers(2, 6)), int(rng.integers(1, 6))
    half = int(rng.integers(0, 2))
    bits = int(rng.choice([1, 2]))
    wrap = int(rng.integers(0, 2))
    kind = RANGE_KINDS[seed % 5]
    if seed == 0:
        lo, hi = -1, 0
    elif kind == "symmetric":
        hi = int(rng.integers(1, 3)) * (1 + half)
        lo = -hi
    elif kind == "asymmetric":
        lo = -1 - int(rng.integers(0, 3))
        hi = -lo + 1 + int(rng.integers(0, 2))
    elif kind == "positive":
        lo = 1 + int(rng.integers(0, 20))
        hi = lo + int(rng.integers(1, 4))
    elif kind == "negative":
        hi = -1 - int(rng.integers(0, 20))
        lo = hi - int(rng.integers(1, 4))
    else:
        lo = hi = int(rng.integers(-15, 16))
    table = _table()
    n_distinct = 1 if seed == 0 else int(rng.integers(1, 6))
    cand = [int(s) for s in rng.choice(len(table), n_distinct, replace=False)]
    if seed % 3 == 1 and SBAS_ROW not in cand:
        cand[0] = SBAS_ROW
    sel = list(cand)
    sel.insert(int(rng.integers(0, len(sel) + 1)), cand[int(rng.integers(0, n_distinct))])   # one repeat
    n_cap = 1 if seed == 0 else int(rng.integers(1, 4))
    step = BIN / (1 + half)
    present = [s for s in cand if s != SBAS_ROW] or [0]
    caps = []
    for c in range(n_cap):
        sig = [(int(s), int(rng.integers(0, 16368)), float(rng.uniform(lo - 0.3, hi + 0.3)) * step,
                float(rng.uniform(42, 47)), float(rng.uniform(0, 2 * np.pi)))
               for s in rng.choice(present, min(len(present), 1 + c % 2), replace=False)]
        caps.append(synth.make_capture(7200 + 10 * seed + c, M * G, table, sig, sample_bits=bits))
    kw = dict(k_noncoh=M * G, half_bin=half, sample_bits=bits, wrap_mode=wrap, dop_lo=lo, dop_hi=hi)
    return table, kw, M, np.array(sel, np.int32), caps


@pytest.mark.parametrize("seed", range(12))
def test_coherent_sweep(gpu_required, oracle, seed):
    """Every cell of every row of every capture against the float64 reference; a repeated satellite gives bitwise the
    same row."""
    table, kw, M, sel, caps = _sweep_case(seed)
    with F.AcqEngine(table, F.default_params(**kw)) as eng:
        rec, grid = eng.search_coherent(np.concatenate(caps), M, sel=sel, want_grid=True)
        p = eng.params
    assert rec.shape == (len(caps), len(sel)) and grid.shape[2] == M * (kw["dop_hi"] - kw["dop_lo"]) + 1
    worst = Worst("coherent sweep seed %d" % seed)
    for c, cap in enumerate(caps):
        base = CoherentRef(oracle, p, cap, table, int(sel[0]))
        seen = {}
        for i, sat in enumerate(sel):
            sat = int(sat)
            if sat in seen:
                j = seen[sat]
                assert grid[c, i].tobytes() == grid[c, j].tobytes() and rec[c, i].tobytes() == rec[c, j].tobytes()
                continue
            seen[sat] = i
            hs, snr = check_cells(grid[c, i], base.for_sat(sat), M, worst=worst, what="capture %d sat %d" % (c, sat))
            assert np.array_equal(hs, grid_h(p, M))
            check_record(rec[c, i], grid[c, i], hs, snr)
    print(worst)


# ---------------------------------------------------------------- many tiles per persistent CTA
def test_many_tiles_per_cta(gpu_required, oracle):
    """K = 8 (two groups of M = 4) on half-bins over +-10 bins: 161 cells per row, 6 captures x 8 rows = 7728 tiles, more
    than ten rounds per CTA (one CTA per SM), so the pending-cell flush and the group prefixes are reused across tiles.
    Copies of a capture at different positions of the batch, and the same capture searched alone, give bitwise the same
    rows; sampled rows against the reference."""
    nav = S.navstar()
    K, M = 8, 4
    kw = dict(k_noncoh=K, half_bin=1, dop_lo=-20, dop_hi=20)
    sel = np.array([1, 4, 7, 10, 13, 16, 19, 22], np.int32)
    a = synth.make_capture(801, K, nav, [(4, 6000, 3.25 * BIN, 44, 0.5), (19, 100, -7.5 * BIN, 43, 2.0)])
    b = synth.make_capture(802, K, nav, [(1, 16000, 9.6 * BIN, 44, 1.1)])
    c = synth.make_capture(803, K, nav, [(22, 8888, -9.875 * BIN, 45, 2.7), (10, 4321, 0.125 * BIN, 43, 0.1)])
    batch = [a, b, c, a, c, b]
    with F.AcqEngine(nav, F.default_params(**kw)) as eng:
        sm = eng.device_info()["sm_count"]
        rec, grid = eng.search_coherent(np.concatenate(batch), M, sel=sel, want_grid=True)
        alone_r, alone_g = eng.search_coherent(a, M, sel=sel, want_grid=True)
        p = eng.params
    assert len(batch) * len(sel) * grid.shape[2] >= 10 * sm
    for i, j in ((0, 3), (2, 4), (1, 5)):
        assert rec[i].tobytes() == rec[j].tobytes() and grid[i].tobytes() == grid[j].tobytes(), (i, j)
    assert alone_r[0].tobytes() == rec[0].tobytes() and alone_g[0].tobytes() == grid[0].tobytes()
    worst = Worst("coherent, many tiles per CTA")
    for ci, cap, s in ((0, a, 1), (2, c, 7), (1, b, 0)):   # rows 4, 22 and 1: each the strongest signal of its capture
        hs, snr = check_cells(grid[ci, s], CoherentRef(oracle, p, cap, nav, int(sel[s])), M, worst=worst)
        check_record(rec[ci, s], grid[ci, s], hs, snr)
    print(worst)
    assert rec[0, 1]["dop"] == 26 and rec[2, 7]["dop"] == -79 and rec[1, 0]["dop"] == 77, rec[:3, [1, 7, 0]]


# ---------------------------------------------------------------- data-bit edges
@pytest.mark.parametrize("m_coh", [4, 5])
def test_data_bit_edges(gpu_required, oracle, m_coh):
    """K = 20 captures with seeded random +-1 data bits: a bit edge before block s = 1..M-1 of group 1 and one in the
    middle of a block (the edges 20 ms later fall 320 samples before a block boundary).  Every cell of the signal row
    against the reference; the record is the signal's cell; with the edge on a block boundary the peak is within 15 %
    of the bit-free capture's."""
    nav = S.navstar()
    K, M = 20, m_coh
    h = M * 2 + 1
    sig = [(3, 5000, h / M * BIN, 47, 0.4)]
    rng = np.random.default_rng(900 + M)
    edges = [(M + s) * synth.BLOCK_SAMPLES for s in range(1, M)] + [(2 * M + 1) * synth.BLOCK_SAMPLES + 32768]
    caps = [synth.make_capture(91, K, nav, sig)]
    for e in edges:
        bits = rng.choice([-1.0, 1.0], 8)
        bits[0] = -bits[-1]   # bit -1 (before the edge) and bit 0 differ
        caps.append(synth.make_capture(91, K, nav, sig, data_bits=bits, bit_edge=e))
    with F.AcqEngine(nav, F.default_params(k_noncoh=K, dop_lo=-3, dop_hi=3)) as eng:
        rec, grid = eng.search_coherent(np.concatenate(caps), M, sel=[3], want_grid=True)
        p = eng.params
    worst = Worst("coherent data-bit edges, M = %d" % M)
    for i, cap in enumerate(caps):
        hs, snr = check_cells(grid[i, 0], CoherentRef(oracle, p, cap, nav, 3), M, worst=worst, what="capture %d" % i)
        check_record(rec[i, 0], grid[i, 0], hs, snr)
        assert (rec[i, 0]["dop"], rec[i, 0]["lag"]) == (h, 1250), (i, rec[i, 0])
    print(worst)
    for i in range(1, M):   # edges on block boundaries
        assert 0.85 <= rec[i, 0]["peak"] / rec[0, 0]["peak"] <= 1.15, (i, rec[i, 0], rec[0, 0])


# ---------------------------------------------------------------- the largest Doppler span
def test_maximum_span(gpu_required, oracle):
    """+-2048 bins at M = 5: 20 481 cells per row.  The first and last five cells and the cells around a signal near
    each end against the reference; the record is the GPU row's best cell and the signal's."""
    nav = S.navstar()
    M = 5
    kw = dict(k_noncoh=M, dop_lo=-2048, dop_hi=2048)
    top, bottom = M * 2048 - 3, -M * 2048 + 4
    caps = synth.make_capture(95, M, nav, [(3, 5000, top / M * BIN, 47, 0.4), (8, 5000, bottom / M * BIN, 47, 1.9)])
    sel = np.array([3, 8], np.int32)
    with F.AcqEngine(nav, F.default_params(**kw)) as eng:
        rec, grid = eng.search_coherent(caps, M, sel=sel, want_grid=True)
        p = eng.params
    n = M * 4096 + 1
    assert grid.shape == (1, 2, n)
    h0 = M * kw["dop_lo"]
    worst = Worst("coherent span +-2048, M = 5")
    for s, h_sig in ((0, top), (1, bottom)):
        g = grid[0, s]
        j = np.unique(np.concatenate([np.arange(5), np.arange(n - 5, n), np.arange(h_sig - h0 - 3, h_sig - h0 + 4)]))
        check_cells(g[j], CoherentRef(oracle, p, caps, nav, int(sel[s])), M, hs=h0 + j, worst=worst)
        b = int(np.argmax(g["snr"]))
        assert rec[0, s]["dop"] == h0 + b == h_sig and rec[0, s]["lag"] == g["lag"][b] == 1250, (s, rec[0, s], b)
    print(worst)


# ---------------------------------------------------------------- the launch split of k_coh_variants
def test_launch_split_of_the_variants(gpu_required, oracle):
    """test_gpu_limits' batch of 33 000 block rows (K = 3) at M = 3, F = 3: k_coh_variants runs on a grid split at
    32 768 rows and forms the sub-bin variants at (row0 + blockIdx.y) mod K.  M = 1 is bitwise acq_search_grid; at M = 3
    every copy of a distinct capture is bitwise every other copy on both sides of the split, and the straddling
    capture and one past the split match the reference.  By ensure_scratch, x2 and the spectra take 2 x 33 000 x 3 x
    128 KiB = 26 GB of device memory (computed, not measured)."""
    nav = S.navstar()
    sel = np.array([3, 17, 25], np.int32)
    kw = dict(dop_lo=-2, dop_hi=2, k_noncoh=SPLIT_K)
    _, caps = split_batch(nav, sel)
    idx = np.arange(SPLIT_CAPTURES) % SPLIT_DISTINCT
    with F.AcqEngine(nav, F.default_params(**kw)) as eng:
        r0, g0 = eng.search(caps.reshape(-1), sel=sel, want_grid=True)
        r1, g1 = eng.search_coherent(caps.reshape(-1), 1, sel=sel, want_grid=True)
        assert r1.tobytes() == r0.tobytes() and g1.tobytes() == g0.tobytes()
        del r0, g0, r1, g1
        rec, grid = eng.search_coherent(caps.reshape(-1), 3, sel=sel, want_grid=True)
        p = eng.params
    rb = rec.view(np.uint8).reshape(SPLIT_CAPTURES, -1)
    gb = grid.view(np.uint8).reshape(SPLIT_CAPTURES, -1)
    assert np.array_equal(rb, rb[idx]) and np.array_equal(gb, gb[idx])
    worst = Worst("coherent launch split")
    for c in (SPLIT_STRADDLE, SPLIT_PAST):
        base = CoherentRef(oracle, p, caps[c], nav, int(sel[0]))
        for s, sat in enumerate(sel):
            hs, snr = check_cells(grid[c, s], base.for_sat(int(sat)), 3, worst=worst)
            check_record(rec[c, s], grid[c, s], hs, snr)
    print(worst)
