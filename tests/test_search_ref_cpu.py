"""CPU side of the precision tier (tests/search_ref.py): the float64 reference against the fp32 oracle's own search cells
and lag profiles at the tight tolerances, against the float64 CoherentRef, and the tolerances against operands rounded
to fp16 precision.  Passing the first shows that fp32 arithmetic can meet the tolerances the GPU tests hold the engine
to."""
import numpy as np
import pytest

from flydog_sdr_gps_b200 import engine, synth
from flydog_sdr_gps_b200 import sats as S

from coherent_ref import CoherentRef
from profile_ref import orc_profile
from search_ref import PEAK_RTOL, SearchRef, Worst, check_cells, check_profile

BIN = engine.BIN_HZ

CASES = {
    # (table, params, signals, sel, sample_bits, code-Doppler capture)
    # row 30's negative bins read row 31, row 31's the zeros after the table
    "ca_k1_reference_wrap": ("nav", dict(), [(3, 2000, 5.4 * BIN, 47, 0.3), (31, 9000, -11.2 * BIN, 47, 1.0)],
                             [3, 30, 31], 1, False),
    "ca_k1_circular_wrap": ("nav", dict(wrap_mode=1), [(30, 700, -8.0 * BIN, 47, 0.3)], [30, 31], 1, False),
    "half_bins": ("nav", dict(half_bin=1, dop_lo=-13, dop_hi=12), [(5, 4004, 2.5 * BIN, 46, 0.5)], [5, 12], 1, False),
    # s(2, h) = round(2 h / 385) is -1 from h = -97 down: shifted and unshifted blocks in one row
    "k3_code_doppler": ("nav", dict(k_noncoh=3, code_doppler=1, dop_lo=-104, dop_hi=-92),
                        [(8, 640, -98.3 * BIN, 45, 2.0)], [8, 3], 1, True),
    "sample_bits_2": ("nav", dict(sample_bits=2), [(12, 333, -3.0 * BIN, 46, 0.7)], [12, 13], 2, False),
    "e1b_k1": ("e1b", dict(dop_lo=-6, dop_hi=5), [(1, 30001, -3.0 * BIN, 48, 0.1)], [1, 4], 1, False),
    "e1b_k4": ("e1b", dict(k_noncoh=4, dop_lo=-3, dop_hi=3), [(1, 30000, -2.0 * BIN, 42, 0.4)], [1, 4], 1, False),
    "k255_one_row": ("nav", dict(k_noncoh=255, dop_lo=-1, dop_hi=1), [(4, 2345, 0.3 * BIN, 30, 0.7)], [4], 1, False),
}


def _case(name):
    which, kw, sig, sel, bits, cd = CASES[name]
    table = S.navstar() if which == "nav" else S.e1b(range(1, 6))
    K = kw.get("k_noncoh", 1)
    return table, kw, synth.make_capture(17, K, table, sig, sample_bits=bits, code_doppler=cd), sel


@pytest.mark.parametrize("name", sorted(CASES))
def test_oracle_meets_the_tolerances(oracle, name):
    """The fp32 oracle's cells at every Doppler index of each row, and its lag profile at each row's best cell, against
    the float64 reference at the tolerances the GPU tests use."""
    table, kw, cap, sel = _case(name)
    p = oracle.default_params(**kw)
    _, grid = oracle.search(cap, table, sel=sel, params=p, want_grid=True)
    ref = SearchRef(oracle, p, cap, table)
    worst = Worst("oracle " + name)
    for s, sat in enumerate(sel):
        cells = ref.cells(sat)
        check_cells(grid[s], cells, worst, "%s sat %d" % (name, sat))
        j = int(np.argmax(cells[3]))
        check_profile(orc_profile(oracle, p, cap, table, sat, int(cells[0][j])), cells[5][j], worst, name)
    print(worst)


def test_two_float64_constructions_agree(oracle):
    """C/A K > 1 on full bins: SearchRef's power is CoherentRef's non-coherent power to 1e-12, at negative bins that read
    the next row and the last row's zeros too."""
    nav = S.navstar()
    p = oracle.default_params(k_noncoh=4, dop_lo=-7, dop_hi=6)
    cap = synth.make_capture(23, 4, nav, [(4, 2345, -2.5 * BIN, 46, 0.7)])
    ref = SearchRef(oracle, p, cap, nav)
    base = CoherentRef(oracle, p, cap, nav, 4)
    for sat in (4, 30, 31):
        coh = base.for_sat(sat)
        for h in range(p.dop_lo, p.dop_hi + 1):
            a, b = ref.power(sat, h), coh.power(h, 1, "noncoh")
            assert np.max(np.abs(a - b)) <= 1e-12 * b.max(), (sat, h)


def _mantissa10(z):
    """z with real and imaginary parts rounded to fp32 and then to a 10-bit mantissa (fp16 precision, fp32 range)."""
    def rnd(x):
        u = np.ascontiguousarray(x, np.float32).view(np.uint32)
        return ((u + np.uint32(0x1000)) & np.uint32(0xFFFFE000)).view(np.float32).astype(np.float64)
    return rnd(z.real) + 1j * rnd(z.imag)


class _Fp16Operands(SearchRef):
    """SearchRef with both operands of the product at fp16 precision."""

    def spectra(self, v):
        fresh = v not in self._D
        D = super().spectra(v)
        if fresh:
            D = self._D[v] = _mantissa10(D)
        return D

    def codes(self, sat):
        fresh = sat not in self._C
        C = super().codes(sat)
        if fresh:
            C = self._C[sat] = tuple(_mantissa10(c) for c in C)
        return C


@pytest.mark.parametrize("which", ["ca", "e1b"])
def test_tolerances_reveal_fp16_operands(oracle, which):
    """Operands at fp16 precision move at least one peak by more than 5 PEAK_RTOL: a search with them cannot pass."""
    if which == "ca":
        table, sel = S.navstar(), [5, 9]
        sig = [(5, 4004, 3 * BIN, 45, 0.3)]
    else:
        table, sel = S.e1b([3, 11, 19]), [0, 1]
        sig = [(0, 30000, -2 * BIN, 45, 0.4)]
    p = oracle.default_params(dop_lo=-6, dop_hi=6)
    cap = synth.make_capture(5, 1, table, sig)
    exact, rounded = SearchRef(oracle, p, cap, table), _Fp16Operands(oracle, p, cap, table)
    moved = max(np.max(np.abs(rounded.cells(sat)[1] / exact.cells(sat)[1] - 1)) for sat in sel)
    assert moved > 5 * PEAK_RTOL, moved
