"""Reference side of the coherent-search tests (acq_search_coherent): the power vectors and cells of a coherent search,
rebuilt in numpy from the oracle's exported stages -- capture baseband, code baseband, the row addressing of its
Correlate restatement (tests/profile_ref.py) -- with every FFT, the sub-bin rotation, the block phases theta_j and the
data-bit hypotheses in float64.  The oracle itself knows nothing of coherent sums."""
import numpy as np

from profile_ref import block_lags, code_row, code_spectra64

N = 16384
LAGS_L1 = 4092


def grid_h(params, m_coh):
    """Doppler indices of a coherent row: M dop_lo .. M dop_hi (1/F-bin steps, F = M (1 + half_bin))."""
    return np.arange(m_coh * params.dop_lo, m_coh * params.dop_hi + 1)


def split_h(h, F):
    """(d, v): integer bin floor(h / F) and sub-bin variant h - F d."""
    d = h // F
    return d, h - F * d


def theta(j, d, v, F, sign16=-1):
    """Phase that puts block j of a group back on the carrier phase of the group's first block, in radians:
    2 pi j (v / F - 16 d / N).  sign16 = +1 gives the sum with the wrong sign on the alignment term (tests only)."""
    return 2.0 * np.pi * j * (v / F + sign16 * 16.0 * d / N)


class CoherentRef:
    """One capture and one satellite of an engine's parameters.  power(h, m_coh, mode) is P[n] over the 4092 lags:
       mode "coherent"  : sum over groups of max over the M data-bit hypotheses |2 S_s - T|^2 (the search's statistic)
       mode "single"    : sum over groups of |T|^2 only (no bit hypothesis)
       mode "noncoh"    : sum over blocks of |r'_b|^2 at the same (d, v) (no phase alignment at all)"""

    def __init__(self, O, params, capture, sats, sat):
        self.O, self.p, self.sats, self.sat = O, params, sats, sat
        self.K = int(params.k_noncoh)
        bits = int(params.sample_bits) or 1
        bb = O.block_bytes(bits)
        cap = np.ascontiguousarray(capture, np.uint8).reshape(-1)
        self.x = [O.capture_baseband(cap[b * bb:(b + 1) * bb], half_rot=0, sample_bits=bits).astype(np.complex128)
                  for b in range(self.K)]
        self.C, self.nxt = code_spectra64(O, sats, sat)
        self._D = {}
        self.n = np.arange(N)

    def for_sat(self, sat):
        """The reference of another satellite on the same capture, sharing its block basebands and spectra."""
        other = object.__new__(type(self))
        other.__dict__.update(self.__dict__)
        other.sat = sat
        other.C, other.nxt = code_spectra64(self.O, self.sats, sat)
        return other

    def spectrum(self, b, v, F):
        key = (b, v, F)
        if key not in self._D:
            rot = np.exp(-2j * np.pi * v * self.n / (F * N)) if v else 1.0
            self._D[key] = np.fft.fft(self.x[b] * rot)
        return self._D[key]

    def lags(self, b, d, v, F):
        """r'_b over the 4092 lags: r_b[(n + 16 b) mod N] (no shift for K = 1, as the search)."""
        code = code_row(self.C, self.nxt, d, self.p.wrap_mode == self.O.WRAP_REFERENCE)
        r = np.fft.ifft(np.conj(self.spectrum(b, v, F)) * code) * N
        return r[block_lags(LAGS_L1, b, 0, self.K, 0, False)]

    def power(self, h, m_coh, mode="coherent", sign16=-1):
        M = int(m_coh)
        F = M * (1 + int(self.p.half_bin))
        d, v = split_h(int(h), F)
        P = np.zeros(LAGS_L1)
        for g in range(self.K // M):
            T = np.zeros(LAGS_L1, np.complex128)
            S = [np.zeros(LAGS_L1, np.complex128)]   # S_0 = 0: "no change" is |T|^2
            for j in range(M):
                r = self.lags(g * M + j, d, v, F)
                if mode == "noncoh":
                    P += np.abs(r) ** 2
                    continue
                if j:
                    S.append(T.copy())
                T = T + np.exp(1j * theta(j, d, v, F, sign16)) * r
            if mode == "coherent":
                P += np.max([np.abs(2 * s - T) ** 2 for s in S], axis=0)
            elif mode == "single":
                P += np.abs(T) ** 2
        return P

    def cells(self, m_coh, hs=None, mode="coherent", sign16=-1):
        """(h, peak, noise, snr, lag, P) over the row's Doppler indices (or hs): Correlate's cell rules on P."""
        hs = grid_h(self.p, m_coh) if hs is None else np.asarray(hs)
        P = np.array([self.power(h, m_coh, mode, sign16) for h in hs])
        peak = P.max(axis=1)
        lag = P.argmax(axis=1)
        noise = P.mean(axis=1)
        return hs, peak, noise, peak / noise, lag, P
