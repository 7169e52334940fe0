"""CPU side of the coherent hand-off (acq_refine_coherent*, acq_profile_coherent*): the float64 reference of
tests/coherent_handoff_ref.py against RefineRef at M = 1, and the phase convention of its group sums pinned by strong
signals at known Doppler offsets between grid points."""
import numpy as np
import pytest

from flydog_sdr_gps_b200 import engine, synth
from flydog_sdr_gps_b200 import sats as S

from coherent_handoff_ref import CoherentHandoffRef
from refine_ref import RefineRef

BIN = engine.BIN_HZ
SAT = 4
# Offset recovery, in bins of the group's DFT (ACQ_BIN_HZ / M).  The three-point estimator of this reference recovers
# the injected offsets of the sweep below to 0.085 bin at most (M = 2 at +-0.4 bin; 0.03 at M = 5): a bias of the
# estimator on these 1-bit captures, not noise (60 dB-Hz).  The tolerance keeps a 1.75x margin.  With the group-start
# correction's sign flipped the same sweep errs by 0.72 bin, so the tolerance separates the two.
OFFSET_TOL = 0.15
OFFSETS = (-0.4, -0.2, 0.0, 0.2, 0.4)
TAU = 15800   # lag ~3950: the group-start phase 2 pi n_b0 / N is near pi, where a wrong sign shows most


def _ref(oracle, M, half_bin, f_hz, seed=7, **kw):
    p = oracle.default_params(k_noncoh=kw.pop("K", M), half_bin=half_bin)
    cap = synth.make_capture(seed, int(p.k_noncoh), S.navstar(), [(SAT, TAU, f_hz, 60, 0.3)], **kw)
    return CoherentHandoffRef(oracle, p, cap, S.navstar(), SAT)


def _offset_errors(oracle, corr, Ms=(2, 3, 4, 5)):
    """(h0, M, half_bin, offset, error in group bins) over the sweep: grid points at +19 bins on v = 0 (the minus point
    crosses into bin d - 1), at 19 bins - H (v = F - H: the plus point crosses into bin d + 1) and at -19 bins."""
    out = []
    for M in Ms:
        for hb in (0, 1):
            H = 1 + hb
            F = M * H
            for h0 in (19 * F, 19 * F - H, -19 * F):
                for off in OFFSETS:
                    f = (h0 + off * H) * BIN / F
                    ref = _ref(oracle, M, hb, f)
                    n = int(np.argmax(ref.power(h0, M)))
                    r = ref.fine(h0, n, M, corr=corr)[0]
                    out.append((h0, M, hb, off, (r["dop_hz"] - f) / (BIN / M)))
    return out


@pytest.mark.parametrize("half_bin", [0, 1])
def test_m1_equals_refine_ref(oracle, half_bin):
    """At M = 1 the coherent reference is RefineRef.fine: same five points, no rotation, the same phases.  (Odd
    half-bins differ by ~1e-8: RefineRef rotates in the oracle's fp32, CoherentRef in float64.)"""
    nav = S.navstar()
    p = oracle.default_params(k_noncoh=3, half_bin=half_bin)
    cap = synth.make_capture(5, 3, nav, [(SAT, 3000, 3.3 * BIN, 45, 0.2)])
    rr, ch = RefineRef(oracle, p, cap, nav), CoherentHandoffRef(oracle, p, cap, nav, SAT)
    for h in ((3, 4, -20, 20) if not half_bin else (6, 7, -41, 41)):
        for n in (0, 1000, 4091):
            a, b = rr.fine(SAT, h, n), ch.fine(h, n, 1)[0]
            assert abs(a["delta"] - b["delta"]) < 1e-6 and abs(a["eps"] - b["eps"]) < 1e-6, (h, n, a, b)
            assert abs(a["peak"] / b["peak"] - 1) < 1e-6, (h, n)
            assert abs(b["dop_hz"] - (a["c"] + max(-1, min(1, a["delta"]))) * BIN) < 1e-3


def test_offsets_are_recovered(oracle):
    """Strong signals at -0.4 .. +0.4 group bins from a grid point, M = 2..5, full and half bins, near +-19 bins, on
    v = 0 and v = F - H: the refined Doppler is the injected one within OFFSET_TOL group bins."""
    errs = _offset_errors(oracle, corr=-1)
    worst = max(abs(e[-1]) for e in errs)
    assert worst <= OFFSET_TOL, [e for e in errs if abs(e[-1]) > OFFSET_TOL]


def test_flipped_group_start_correction_fails(oracle):
    """The same sweep with e^{+j 2 pi (d' - d) n_b0 / N} in place of e^{-j ...} misses the tolerance."""
    errs = _offset_errors(oracle, corr=+1, Ms=(2, 4))
    assert max(abs(e[-1]) for e in errs) > 2 * OFFSET_TOL


@pytest.mark.parametrize("edge", [1, 2, 3])
def test_data_bit_edge(oracle, edge):
    """M = 4, K = 8, a data-bit sign change before block `edge` of the first group: the centre's hypothesis takes the
    edge, and the refined Doppler and code phase stay within the bounds of the edge-free capture."""
    M, hb = 4, 0
    h0 = 19 * M - 1
    for off in (-0.3, 0.3):
        f = (h0 + off) * BIN / M
        clean = _ref(oracle, M, hb, f, K=2 * M)
        edged = _ref(oracle, M, hb, f, K=2 * M, data_bits=[1, -1], bit_edge=edge * 65536)
        n = int(np.argmax(clean.power(h0, M)))
        assert int(np.argmax(edged.power(h0, M))) == n
        a, b = clean.fine(h0, n, M)[0], edged.fine(h0, n, M)[0]
        assert abs((b["dop_hz"] - f) / (BIN / M)) <= OFFSET_TOL, (edge, off, b["dop_hz"], f)
        assert abs(b["code_fs"] - a["code_fs"]) <= 0.25, (edge, off, a["code_fs"], b["code_fs"])
        # without the hypothesis the edge group would cancel: the chosen one recovers the clean peak's size
        assert b["peak"] > 0.5 * a["peak"], (edge, b["peak"], a["peak"])
