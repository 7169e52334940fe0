"""CPU side of the coherent searches' precision tier: a single-precision emulation of CoherentRef -- fp32 FFTs
(scipy.fft keeps complex64 in single precision), fp32 sub-bin rotation, block phases, data-bit prefixes S_s and powers
-- against the float64 CoherentRef at search_ref's tolerances with a 3x margin, over M = 2..5, half-bins, K = 255 and
the +-2048-bin span.  Passing shows that fp32 arithmetic meets the tolerances test_gpu_coherent*, which hold the
coherent kernels to them, use.  Capture spectra at fp16 precision (10-bit mantissa) must not."""
import numpy as np
import pytest
import scipy.fft

from flydog_sdr_gps_b200 import engine, synth
from flydog_sdr_gps_b200 import sats as S

from coherent_ref import LAGS_L1, N, CoherentRef, grid_h, split_h, theta
from profile_ref import block_lags, code_row
from search_ref import PEAK_RTOL, Worst, check_cells
from test_search_ref_cpu import _mantissa10

BIN = engine.BIN_HZ


class CoherentRef32(CoherentRef):
    """CoherentRef with every step in single precision."""

    def __init__(self, *a):
        super().__init__(*a)
        self.x = [x.astype(np.complex64) for x in self.x]
        self._codes32()

    def _codes32(self):
        def fft(s):
            return scipy.fft.fft(self.O.code_baseband(self.sats[s])) if s < len(self.sats) else np.zeros(N, np.complex64)
        self.C, self.nxt = fft(self.sat), fft(self.sat + 1)

    def for_sat(self, sat):
        other = super().for_sat(sat)
        other._codes32()
        return other

    def spectrum(self, b, v, F):
        key = (b, v, F)
        if key not in self._D:
            rot = np.exp(-2j * np.pi * v * self.n / (F * N)).astype(np.complex64) if v else np.complex64(1)
            self._D[key] = self.quantise(scipy.fft.fft(self.x[b] * rot))
        return self._D[key]

    def quantise(self, D):
        return D

    def lags(self, b, d, v, F):
        code = code_row(self.C, self.nxt, d, self.p.wrap_mode == self.O.WRAP_REFERENCE)
        r = scipy.fft.ifft(np.conj(self.spectrum(b, v, F)) * code, norm="forward")
        return r[block_lags(LAGS_L1, b, 0, self.K, 0, False)]

    def power(self, h, m_coh, mode="coherent", sign16=-1):
        assert mode == "coherent"
        M = int(m_coh)
        F = M * (1 + int(self.p.half_bin))
        d, v = split_h(int(h), F)
        P = np.zeros(LAGS_L1, np.float32)
        for g in range(self.K // M):
            T = np.zeros(LAGS_L1, np.complex64)
            Ss = [T.copy()]
            for j in range(M):
                r = self.lags(g * M + j, d, v, F)
                if j:
                    Ss.append(T.copy())
                T = T + np.complex64(np.exp(1j * theta(j, d, v, F))) * r
            P = P + np.max([np.abs(np.complex64(2) * s - T).astype(np.float32) ** 2 for s in Ss], axis=0)
        return P


class Fp16Spectra(CoherentRef32):
    """... with the capture spectra stored at fp16 precision (10-bit mantissa, fp32 range)."""

    def quantise(self, D):
        return _mantissa10(D).astype(np.complex64)


CASES = {
    # (params, M, signals, sel, hs: None for the whole row or (first, last) indices relative to M dop_lo)
    "m2_k4": (dict(k_noncoh=4, dop_lo=-3, dop_hi=2), 2, [(9, 3000, 1.5 * BIN, 41, 0.9)], [9, 14], None),
    "m3_half_bins": (dict(k_noncoh=3, half_bin=1, dop_lo=-4, dop_hi=3), 3, [(9, 3000, 7 / 6 * BIN, 41, 0.9)], [9], None),
    "m4_k8_circular": (dict(k_noncoh=8, wrap_mode=1, dop_lo=-2, dop_hi=2), 4, [(30, 700, -1.25 * BIN, 42, 0.3)],
                       [30, 31], None),
    "m5_half_bins_2bit": (dict(k_noncoh=5, half_bin=1, sample_bits=2, dop_lo=-2, dop_hi=2), 5,
                          [(3, 5000, 0.7 * BIN, 44, 0.4)], [3], None),
    "m5_k255": (dict(k_noncoh=255, dop_lo=-1, dop_hi=0), 5, [(4, 2345, -0.4 * BIN, 32, 0.7)], [4], None),
    "m5_span_2048": (dict(k_noncoh=5, dop_lo=-2048, dop_hi=2048), 5, [(3, 5000, 2047.4 * BIN, 47, 0.4)], [3, 31],
                     ((0, 6), (5 * 4096 - 8, 5 * 4096 + 1))),
}


def _case(O, name):
    kw, M, sig, sel, hs = CASES[name]
    nav = S.navstar()
    bits = kw.get("sample_bits", 1)
    cap = synth.make_capture(61, kw["k_noncoh"], nav, sig, sample_bits=bits)
    p = O.default_params(**kw)
    if hs is not None:
        hs = np.concatenate([M * p.dop_lo + np.arange(a, b) for a, b in hs])
    return nav, p, cap, M, sel, hs


@pytest.mark.parametrize("name", sorted(CASES))
def test_fp32_coherent_meets_the_tier_with_margin(oracle, name):
    """Every cell of each row (or of the span's ends) of the fp32 emulation within a third of search_ref's tolerances."""
    nav, p, cap, M, sel, hs = _case(oracle, name)
    worst = Worst("fp32 coherent " + name)
    base, base32 = CoherentRef(oracle, p, cap, nav, sel[0]), CoherentRef32(oracle, p, cap, nav, sel[0])
    for sat in sel:
        ref = base.for_sat(sat).cells(M, hs=hs)
        _, peak, noise, snr, lag, _ = base32.for_sat(sat).cells(M, hs=hs)
        got = np.zeros(peak.size, [("peak", "<f4"), ("noise", "<f4"), ("snr", "<f4"), ("lag", "<i4")])
        got["peak"], got["noise"], got["snr"], got["lag"] = peak, noise, snr, lag
        check_cells(got, ref, worst, "%s sat %d" % (name, sat), margin=3.0)
    print(worst)


def test_fp16_capture_spectra_fail_the_tier(oracle):
    """Capture spectra with a 10-bit mantissa move a coherent peak by more than 5 PEAK_RTOL."""
    nav, p, cap, M, sel, hs = _case(oracle, "m2_k4")
    exact, rounded = CoherentRef(oracle, p, cap, nav, 9), Fp16Spectra(oracle, p, cap, nav, 9)
    moved = np.max(np.abs(rounded.cells(M)[1] / exact.cells(M)[1] - 1))
    assert moved > 5 * PEAK_RTOL, moved
