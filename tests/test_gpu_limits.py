"""GPU suite (-m gpu) at the limits acq_create accepts: the Doppler span of 2048 bins either side (the margin Q of the
extended code rows), K = 255 non-coherent blocks, code-Doppler compensation at its 33 shifted copies per spectrum, and a
batch of more than 32 768 block rows (the front end's launch split).  Each case against the CPU oracle on the same
bytes: records, the whole per-Doppler table, acq_refine against oracle.refine and the float64 RefineRef
(tests/refine_ref.py), and acq_profile against orc_profile."""
import numpy as np
import pytest

import flydog_sdr_gps_b200 as F
from flydog_sdr_gps_b200 import synth
from flydog_sdr_gps_b200 import sats as S

from parity import RTOL, Margins, compare_records
from profile_ref import circular_distance, code_shift, orc_profile, peak2_of
from refine_ref import RefineRef, check_fine
from search_ref import Worst
from test_gpu_parity import _compare_fine

pytestmark = pytest.mark.gpu
BIN = F.BIN_HZ
EXCL = 4


def _thr(table, sel, kw):
    return np.array([kw.get("thr_e1b", 16.0) if table[s][3] == S.E1B else kw.get("thr_l1", 16.0) for s in sel])


def _search_vs_oracle(eng, oracle, table, kw, cap, sel, label):
    """Records and per-Doppler tables of one capture against the oracle, row by row (per-constellation thresholds)."""
    rec, grid = eng.search(cap, sel=sel, want_grid=True)
    orec, ogrid = oracle.search(cap, table, sel=sel, params=oracle.default_params(**kw), want_grid=True)
    assert np.array_equal(rec[0]["sat"], sel)
    m = Margins(label)
    thr = _thr(table, sel, kw)
    for i in range(len(sel)):
        compare_records(rec[0][i:i + 1], orec[i:i + 1], ogrid[i:i + 1], kw["dop_lo"], float(thr[i]),
                        ggrid=grid[0][i:i + 1], max_ties=1, margins=m)
    m.report()
    return rec, orec


def _refine_vs_oracle(eng, oracle, table, kw, cap, rec, rows=None):
    """acq_refine of the last search's records against oracle.refine of the same records (test_gpu_parity's
    tolerances) and against the float64 RefineRef (refine_ref's bound), over `rows` (default: all)."""
    fine = eng.refine(rec)
    oprm = oracle.default_params(**kw)
    ofine = oracle.refine(cap, table, rec[0], params=oprm)
    rows = np.arange(rec.shape[1]) if rows is None else np.asarray(rows)
    if rows.size:
        _compare_fine(fine[0][rows], ofine[rows], rec[0][rows])
        worst = Worst("refine at the limits")
        check_fine(fine[0][rows], rec[0][rows], RefineRef(oracle, oprm, cap, table), worst)
        print(worst)
    return fine


def _profile_vs_oracle(eng, oracle, table, kw, cap, rec):
    """acq_profile of the last search's records against orc_profile (test_gpu_profile's tolerances)."""
    pk, prof = eng.profile(rec, excl=EXCL, want_profile=True)
    off = eng.profile_offsets(1, rec[0]["sat"])
    oprm = oracle.default_params(**kw)
    for i, r in enumerate(rec[0]):
        row = prof[off[i]:off[i + 1]]
        lag = int(r["lag"])
        assert row[lag] == r["peak"] and int(np.argmax(row)) == lag, (i, row[lag], r["peak"])
        P = orc_profile(oracle, oprm, cap, table, int(r["sat"]), int(r["dop"]))
        assert row.size == P.size
        assert np.allclose(row, P, rtol=RTOL, atol=RTOL * P.mean()), (i, np.max(np.abs(row - P)) / P.mean())
        out = circular_distance(row.size, lag) > EXCL
        g = pk[0, i]
        o_peak2, o_lag2, o_ratio, o_noise = peak2_of(P, lag, EXCL)
        assert abs(g["peak2"] - o_peak2) <= RTOL * o_peak2
        assert g["lag2"] == o_lag2 or (out[g["lag2"]] and P[g["lag2"]] >= (1 - RTOL) * o_peak2), (i, g["lag2"], o_lag2)
        assert abs(g["ratio"] - o_ratio) <= 2 * RTOL * o_ratio
        assert abs(g["noise_ex"] - o_noise) <= RTOL * o_noise


# ---------------------------------------------------------------- 1. Doppler span at the limit (|bins| = 2048)
# Signals a fraction of a bin inside each end, so that their records sit on the edge cells dop_lo / dop_hi: a refinement
# there reads code rows d - 1 and d + 1, one bin past the range, which is what the margin Q of the extended rows covers.
SPAN_CASES = {
    "full_bins_2048": (dict(dop_lo=-2048, dop_hi=2048), 2047.8, -2047.8),
    "half_bins_4094": (dict(dop_lo=-4094, dop_hi=4094, half_bin=1), 2046.9, -2046.9),
}


@pytest.mark.parametrize("wrap", [F.WRAP_REFERENCE, F.WRAP_CIRCULAR])
@pytest.mark.parametrize("case", sorted(SPAN_CASES))
def test_doppler_span_at_the_limit(gpu_required, oracle, case, wrap):
    """Rows: C/A 5 (signal at the top end), C/A 9 (signal at the bottom end), C/A 0 (in the reference wrap its negative
    Doppler bins read row 1) and E1B 44, over the largest range acq_create accepts."""
    base, f_hi, f_lo = SPAN_CASES[case]
    kw = dict(base, wrap_mode=wrap)
    table = S.reference_table()
    cap = synth.make_capture(610 + wrap, 1, table, [(5, 4004, f_hi * BIN, 49, 0.4), (9, 9000, f_lo * BIN, 49, 2.1)])
    sel = np.array([5, 9, 0, 44], np.int32)
    with F.AcqEngine(table, F.default_params(**kw)) as eng:
        assert eng.n_dop == kw["dop_hi"] - kw["dop_lo"] + 1
        rec, orec = _search_vs_oracle(eng, oracle, table, kw, cap, sel, "span %s wrap %d" % (case, wrap))
        assert rec[0]["dop"][0] == kw["dop_hi"] and rec[0]["dop"][1] == kw["dop_lo"], rec[0]
        _refine_vs_oracle(eng, oracle, table, kw, cap, rec)
        _profile_vs_oracle(eng, oracle, table, kw, cap, rec)
    with pytest.raises(F.AcqError) as ei:   # one more bin either side is refused
        F.AcqEngine(table, F.default_params(**dict(kw, dop_hi=kw["dop_hi"] + 2)))
    assert ei.value.code == -1


# ---------------------------------------------------------------- 2. K = 255 non-coherent blocks
K_MAX = 255
K255_CASES = {
    # (table, params keywords, sample_bits, sel, signals)
    "ca_1bit": (S.reference_table(), dict(dop_lo=-2, dop_hi=2), 1, [5, 31, 35, 0],
                [(5, 4000, 1.0 * BIN, 38, 0.3), (0, 12000, -1.6 * BIN, 39, 1.0)]),
    "ca_2bit_half_bins": (S.navstar(), dict(dop_lo=-3, dop_hi=1, half_bin=1, sample_bits=2), 2, [7, 2, 19],
                          [(7, 2000, -0.5 * BIN, 38, 0.2), (19, 15000, 0.5 * BIN, 39, 2.0)]),
    "ca_circular": (S.reference_table(), dict(dop_lo=-3, dop_hi=0, wrap_mode=F.WRAP_CIRCULAR), 1, [0, 35, 12],
                    [(0, 333, -2.0 * BIN, 38, 0.9), (12, 8000, -0.8 * BIN, 38, 0.4)]),
    # nine E1B rows x 5 Doppler indices: more tiles than a cluster each, so k_search_e1b_multi runs
    "e1b_multi": (S.e1b([2, 3, 4, 5, 7, 8, 9, 10, 11]), dict(dop_lo=-2, dop_hi=2), 1, list(range(9)),
                  [(1, 30000, 1.0 * BIN, 40, 0.4), (6, 4096, -2.0 * BIN, 40, 1.3)]),
}


@pytest.mark.parametrize("case", sorted(K255_CASES))
def test_k255_blocks(gpu_required, oracle, case):
    """K = 255 (the largest k_noncoh): the front end's block delay 16 (b mod K) reaches 4064 samples and every cell sums
    255 block powers.  Records and whole tables against the oracle, refinement of the detected rows."""
    table, over, bits, sel, sig = K255_CASES[case]
    kw = dict(over, k_noncoh=K_MAX, thr_l1=3.0, thr_e1b=3.0)
    sel = np.array(sel, np.int32)
    cap = synth.make_capture(620 + sorted(K255_CASES).index(case), K_MAX, table, sig, sample_bits=bits)
    with F.AcqEngine(table, F.default_params(**kw)) as eng:
        rec, orec = _search_vs_oracle(eng, oracle, table, kw, cap, sel, "K = 255 %s" % case)
        det = np.nonzero(orec["snr"] >= _thr(table, sel, kw) * (1 + RTOL))[0]
        assert len(det) >= 2, orec
        _refine_vs_oracle(eng, oracle, table, kw, cap, rec, rows=det)


# ---------------------------------------------------------------- 3. code-Doppler compensation at 33 copies
# s(b, h) = round(b h / (385 (1 + half_bin))) reaches smax = 16 in the last block: 2 smax + 1 = 33 = ACQ_MAX_CODE_SHIFTS.
CD_CASES = {
    # (table, K, params keywords, signal row, signal Doppler in bins, sel)
    "ca_k20_full_bins_pos": (S.navstar(), 20, dict(dop_lo=300, dop_hi=320), 4, 318.0, [4, 11]),
    "ca_k20_full_bins_neg": (S.navstar(), 20, dict(dop_lo=-320, dop_hi=-300), 4, -317.0, [4, 11]),
    "ca_k20_half_bins_neg": (S.navstar(), 20, dict(dop_lo=-640, dop_hi=-600, half_bin=1), 9, -318.5, [9, 0]),
    "e1b_k6_full_bins": (S.e1b([3, 11, 19]), 6, dict(dop_lo=-1270, dop_hi=-1262), 1, -1266.0, [1, 2]),
}


@pytest.mark.parametrize("case", sorted(CD_CASES))
def test_code_doppler_at_33_copies(gpu_required, oracle, case):
    """code_doppler at the largest number of shifted copies acq_create accepts; one Doppler index further out needs 35
    and is ACQ_ERR_UNSUPPORTED.  Captures stretched by their carrier offsets; search, refine and profile against the
    oracle and orc_profile."""
    table, K, over, sat, f_bins, sel = CD_CASES[case]
    hb = over.get("half_bin", 0)
    kw = dict(over, k_noncoh=K, code_doppler=1, thr_l1=3.0, thr_e1b=3.0)
    smax = max(abs(code_shift(K - 1, kw["dop_lo"], hb)), abs(code_shift(K - 1, kw["dop_hi"], hb)))
    assert 2 * smax + 1 == 33
    far = kw["dop_hi"] if abs(kw["dop_hi"]) > abs(kw["dop_lo"]) else kw["dop_lo"]
    step = 1 if far > 0 else -1
    while abs(code_shift(K - 1, far, hb)) == smax:
        far += step
    with pytest.raises(F.AcqError) as ei:
        F.AcqEngine(table, F.default_params(**dict(kw, dop_lo=min(far, kw["dop_lo"]), dop_hi=max(far, kw["dop_hi"]))))
    assert ei.value.code == -4 and "35" in str(ei.value)
    sel = np.array(sel, np.int32)
    period = 65472 if table[sat][3] == S.E1B else 16368
    cap = synth.make_capture(630 + K, K, table, [(sat, period // 3, f_bins * BIN, 44 if K == 20 else 47, 0.6)],
                             code_doppler=True)
    with F.AcqEngine(table, F.default_params(**kw)) as eng:
        rec, orec = _search_vs_oracle(eng, oracle, table, kw, cap, sel, "code_doppler %s" % case)
        assert rec[0]["dop"][0] == round(f_bins * (1 + hb)) and rec[0]["snr"][0] >= 3.0, rec[0]
        _refine_vs_oracle(eng, oracle, table, kw, cap, rec)
        _profile_vs_oracle(eng, oracle, table, kw, cap, rec)


# ---------------------------------------------------------------- 4. more than 32 768 block rows in one call
# The front end runs on a grid of at most 32 768 block rows per launch and passes the first row (row0) of each launch:
# block b of a capture is delayed by 16 ((row0 + blockIdx.y) mod K) samples.  K = 3 and 11 000 captures = 33 000 rows;
# capture 10 922 owns rows 32 766..32 768 and so straddles the split, and since 32 768 mod 3 != 0 a launch that lost row0
# would delay every later block by the wrong amount.  By ensure_scratch, x2 and the capture spectra of this call take
# 2 x 33 000 x 128 KiB = 8.7 GB of device memory (computed, not measured).
SPLIT_K, SPLIT_CAPTURES, SPLIT_DISTINCT = 3, 11_000, 8
SPLIT_STRADDLE, SPLIT_PAST = 10_922, 10_925


def split_batch(table, sel):
    """(distinct captures [8, K*8192], the batch [11 000, K*8192]): capture c of the batch is distinct capture c % 8."""
    distinct = np.stack([synth.make_capture(700 + i, SPLIT_K, table,
                                            [(int(sel[i % len(sel)]), 1000 + 977 * i, (i % 5 - 2) * 0.9 * BIN, 46, 0.3 * i),
                                             (int(sel[(i + 1) % len(sel)]), 13000 - 555 * i, (2 - i % 4) * 0.6 * BIN, 44, 1.0)])
                         for i in range(SPLIT_DISTINCT)])
    return distinct, distinct[np.arange(SPLIT_CAPTURES) % SPLIT_DISTINCT]


def test_launch_split_past_32768_block_rows(gpu_required, oracle):
    """Host and device forms over 33 000 block rows: every copy of a distinct capture gives bitwise the records and
    per-Doppler table of every other copy, on both sides of the split; the straddling capture and one past the split
    match the oracle."""
    import torch
    assert SPLIT_STRADDLE * SPLIT_K < 32768 < (SPLIT_STRADDLE + 1) * SPLIT_K and 32768 % SPLIT_K
    table = S.navstar()
    sel = np.array([3, 17, 25], np.int32)
    kw = dict(dop_lo=-2, dop_hi=2, k_noncoh=SPLIT_K, thr_l1=8.0)
    distinct, caps = split_batch(table, sel)
    idx = np.arange(SPLIT_CAPTURES) % SPLIT_DISTINCT
    with F.AcqEngine(table, F.default_params(**kw)) as eng:
        rec, grid = eng.search(caps.reshape(-1), sel=sel, want_grid=True)
        assert rec.shape == (SPLIT_CAPTURES, len(sel))
        rb = rec.view(np.uint8).reshape(SPLIT_CAPTURES, -1)
        gb = grid.view(np.uint8).reshape(SPLIT_CAPTURES, -1)
        assert np.array_equal(rb, rb[idx]) and np.array_equal(gb, gb[idx])
        d_in = torch.from_numpy(caps.reshape(-1)).cuda()
        d_out = torch.zeros(rec.nbytes, dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()
        eng.search_device(d_in.data_ptr(), d_out.data_ptr(), SPLIT_CAPTURES, sel=sel)
        torch.cuda.synchronize()
        assert d_out.cpu().numpy().tobytes() == rec.tobytes()
        del d_in, d_out
    m = Margins("launch split, captures %d and %d" % (SPLIT_STRADDLE, SPLIT_PAST))
    for c in (SPLIT_STRADDLE, SPLIT_PAST):
        orec, ogrid = oracle.search(caps[c], table, sel=sel, params=oracle.default_params(**kw), want_grid=True)
        compare_records(rec[c], orec, ogrid, kw["dop_lo"], kw["thr_l1"], ggrid=grid[c], max_ties=1, margins=m)
    m.report()
