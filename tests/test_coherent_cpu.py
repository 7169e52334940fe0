"""CPU side of the coherent search (acq_search_coherent): exports, the argument errors decided before the engine is read,
the reference (tests/coherent_ref.py) at M = 1 against the oracle's own search cells, and the synthetic captures'
default bytes."""
import ctypes as C
import hashlib

import numpy as np
import pytest

from flydog_sdr_gps_b200 import _lib, engine, synth
from flydog_sdr_gps_b200 import sats as S

from coherent_ref import CoherentRef, grid_h

BIN = engine.BIN_HZ


def test_exports():
    L = _lib.load()
    for name in ("acq_search_coherent", "acq_search_coherent_device"):
        assert name in _lib.exported_symbols() and hasattr(L, name)
    assert hasattr(engine.AcqEngine, "search_coherent") and hasattr(engine.AcqEngine, "search_coherent_device")


def test_argument_errors_before_the_engine():
    """A NULL engine and an m_coh outside 1..ACQ_COH_MAX (5) are ACQ_ERR_ARG (-1) before the engine is read."""
    L = _lib.load()
    buf = np.zeros(8192, np.uint8)
    out = np.zeros(4, engine.RECORD_DTYPE)
    p, o = buf.ctypes.data, out.ctypes.data
    assert L.acq_search_coherent(None, p, 1, None, 0, 1, o, None) == -1
    assert b"engine is NULL" in L.acq_last_error()
    assert L.acq_search_coherent_device(None, p, 1, None, 0, 1, o, None) == -1
    assert b"engine is NULL" in L.acq_last_error()
    fake = C.c_void_p(o)   # any non-NULL handle: the m_coh range is checked before the engine is read
    for m in (0, -1, 6, 100):
        assert L.acq_search_coherent(fake, p, 1, None, 0, m, o, None) == -1
        assert b"m_coh=%d outside 1..5" % m in L.acq_last_error()
        assert L.acq_search_coherent_device(fake, p, 1, None, 0, m, o, None) == -1
        assert b"m_coh=%d outside 1..5" % m in L.acq_last_error()


M1_CASES = {
    "full_bins_reference_wrap_k1": (dict(), 1, 1),
    "half_bins_k4": (dict(half_bin=1, k_noncoh=4, dop_lo=-9, dop_hi=7), 4, 1),
    "circular_wrap_k4": (dict(wrap_mode=1, k_noncoh=4, dop_lo=-12, dop_hi=3), 4, 1),
    "two_bit_half_bins": (dict(sample_bits=2, half_bin=1, dop_lo=-8, dop_hi=8), 1, 2),
    # the shapes of the GPU limit tests: K = 255, the circular wrap on 2-bit samples, both ends of the +-2048-bin span
    "k255_narrow": (dict(k_noncoh=255, dop_lo=-1, dop_hi=1), 255, 1),
    "circular_wrap_two_bit_k3": (dict(wrap_mode=1, sample_bits=2, k_noncoh=3, dop_lo=-6, dop_hi=4), 3, 2),
    "span_top_full_bins": (dict(dop_lo=2042, dop_hi=2048), 1, 1),
    "span_bottom_half_bins": (dict(half_bin=1, dop_lo=-4094, dop_hi=-4087), 1, 1),
}


@pytest.mark.parametrize("case", sorted(M1_CASES))
def test_reference_m1_is_the_oracle_search(oracle, case):
    """At M = 1 the reference's cells are the oracle's search(..., want_grid=True) cells: peak, noise and snr within
    float32 rounding, and the lag wherever the reference's own runner-up lag is not within that rounding."""
    kw, K, bits = M1_CASES[case]
    table = S.navstar()
    params = oracle.default_params(**kw)
    sig = [(4, 2345, -2.5 * BIN, 46, 0.7), (11, 15000, 3.0 * BIN, 44, 2.0)]
    cap = synth.make_capture(31, K, table, sig, sample_bits=bits)
    sel = [4, 11, 20, 0]   # 0: wraps into row 1 at negative Doppler in the reference wrap
    _, grid = oracle.search(cap, table, sel=sel, params=params, want_grid=True)
    base = CoherentRef(oracle, params, cap, table, sel[0])
    for s, sat in enumerate(sel):
        hs, peak, noise, snr, lag, P = base.for_sat(sat).cells(1)
        assert np.array_equal(hs, grid_h(params, 1))
        g = grid[s]
        np.testing.assert_allclose(peak, g["peak"], rtol=2e-5)
        np.testing.assert_allclose(noise, g["noise"], rtol=2e-5)
        np.testing.assert_allclose(snr, g["snr"], rtol=2e-5)
        at_oracle_lag = P[np.arange(len(hs)), g["lag"]]
        assert np.all((lag == g["lag"]) | (at_oracle_lag >= peak * (1 - 1e-4))), (case, sat)


# sha256 of the bytes of default make_capture calls (no data bits), taken before the data-bit option existed
DEFAULT_DIGESTS = [
    "1e8e029df04fc7f958ab5969ffda581b2705f86e642405a9339468e81d5cad27",
    "d0f25db642b2807f941bfee767ca1b0253b9a5c31366d1c058c00e888f3a3ba7",
    "f185980ecfcff054d756cef30082a3c6bee55167e63d481a9ce3dd133e880bd7",
]


def _default_calls():
    t, nav = S.reference_table(), S.navstar()
    return [
        synth.make_capture(4242, 1, t, [(2, 4000, 4 * BIN, 48, 1.0), (10, 8188, -10 * BIN, 47, 2.0), (44, 30000, -6 * BIN, 47, 0.4)]),
        synth.make_capture(9, 2, nav, [(5, 777, -3.3 * BIN, 45, 0.2)], sample_bits=2),
        synth.make_capture(10, 3, nav, [(7, 123, 17.5 * BIN, 44, 2.2)], code_doppler=True),
    ]


def test_default_capture_bytes_unchanged():
    assert [hashlib.sha256(c.tobytes()).hexdigest() for c in _default_calls()] == DEFAULT_DIGESTS


def test_data_bits_modulate_the_signal():
    """All-ones bits give the default bytes; a sign change at a block boundary flips the signal's sign from there on, so
    the block correlations of the reference change sign against each other."""
    nav = S.navstar()
    sig = [(5, 777, -3.0 * BIN, 60, 0.2)]
    base = synth.make_capture(9, 2, nav, sig)
    assert np.array_equal(synth.make_capture(9, 2, nav, sig, data_bits=[1, 1]), base)
    flipped = synth.make_capture(9, 2, nav, sig, data_bits=[1, -1], bit_edge=65536 - synth.BIT_SAMPLES)
    assert np.array_equal(flipped[:8192], base[:8192]) and not np.array_equal(flipped[8192:], base[8192:])
