"""CPU suite for the aided search (acq_search_aided / acq_search_aided_device): exported by the library and the binding,
and its argument errors are reported before any device work -- no GPU needed."""
import numpy as np

from flydog_sdr_gps_b200 import _lib

ENTRY_POINTS = ("acq_search_aided", "acq_search_aided_device")


def test_both_entry_points_are_exported_and_bound():
    L = _lib.load()
    names = _lib.exported_symbols()
    for n in ENTRY_POINTS:
        assert n in names and hasattr(L, n)


def _call(L, name, eng, center, half_width):
    cap = np.zeros(8192, np.uint8)
    out = np.zeros(64, np.uint8)
    c = center.ctypes.data if center is not None else None
    # the last argument is the grid (host form) or the stream (device form): NULL for both
    return getattr(L, name)(eng, cap.ctypes.data, 1, None, 0, c, half_width, out.ctypes.data, None)


def test_argument_errors_without_gpu():
    """A NULL engine, a NULL dop_center, a negative half_width and a window wider than any engine's Doppler range are
    ACQ_ERR_ARG (-1) with their own text."""
    L = _lib.load()
    center = np.zeros(64, np.int32)
    for name in ENTRY_POINTS:
        assert _call(L, name, None, center, 2) == -1
        assert b"engine is NULL" in L.acq_last_error()
        assert _call(L, name, None, None, 2) == -1
        assert b"dop_center is NULL" in L.acq_last_error()
        assert _call(L, name, None, center, -1) == -1
        assert b"half_width must be >= 0" in L.acq_last_error()
        # W = 2 * 5000 + 1 exceeds n_dop of every engine (|Doppler index| <= 4094); also keeps 2 * half_width + 1 from overflowing
        for hw in (5000, 2 ** 31 - 1):
            assert _call(L, name, None, center, hw) == -1
            assert b"exceeds n_dop" in L.acq_last_error()


def test_window_base_rule():
    """The window rule of the header, restated: lo = clamp(center - half_width, dop_lo, dop_hi - 2 half_width); every row
    gets W indices inside the range whatever its centre (what the GPU tests check the kernels against)."""
    def lo(c, hw, dlo, dhi):
        return min(max(c - hw, dlo), dhi - 2 * hw)
    for dlo, dhi in ((-20, 20), (-7, 30), (3, 3), (-80, 80)):
        for hw in range(0, (dhi - dlo) // 2 + 1):
            for c in (-2 ** 31, dlo - 5, dlo, 0, dhi, dhi + 5, 2 ** 31 - 1):
                b = lo(c, hw, dlo, dhi)
                assert dlo <= b and b + 2 * hw <= dhi
                if dlo + hw <= c <= dhi - hw:
                    assert b == c - hw
