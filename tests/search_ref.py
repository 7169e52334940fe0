"""Float64 reference of the non-coherent search (acq_search, acq_search_grid, acq_profile), and the precision tier of the
tests built on it.

SearchRef rebuilds the power vector of every search cell -- the sum over the K blocks of |IFFT(conj(D_b) * code row)|^2
at the row's lags -- with every FFT and product in float64.  Its inputs are the oracle's fp32 capture baseband, which the
engine's front end matches to the bit (half-bin rotation and 2-bit samples included), and its code baseband.  The
addressing is correlate_one's, from profile_ref (code_row, block_lags), shared with orc_profile and CoherentRef.

parity.RTOL (1e-3 against the fp32 oracle) decides whether the engine computes the reference's search.  The tolerances
here decide whether it computes it at the precision fp32 arithmetic reaches, which is some 100 times tighter.

Error model.  Every stage of the engine rounds in fp32 (unit roundoff u = 6e-8): the spectra, their product and the
16384-point inverse FFT leave an absolute error on each lag value r[n] that scales with the transform's RMS, sqrt(m)
(m: the row's mean power).  A power P = |r|^2 is then off by about c u (2 |r| sqrt(m) + m), so |error| / sqrt(P m + m^2)
is a constant of the arithmetic, and PROFILE_TAU bounds it.  A peak (P >> m) is off by less than that relative to
itself.  The noise, a mean over L lags, also carries the rounding of its own fp32 sum.  The fp32 oracle, whose sums run
in sequence, against this reference on the CPU, largest relative errors:
    C/A K = 1, 4 rows x 41 bins     peak 5.6e-7   noise 2.6e-6   snr 2.6e-6
    C/A K = 4, half-bins            peak 3.4e-7   noise 2.8e-6   snr 2.8e-6
    E1B K = 1                       peak 3.3e-7   noise 5.7e-6   snr 5.7e-6
    E1B K = 4                       peak 2.5e-7   noise 4.7e-6   snr 5.0e-6
    lag profiles                    |P32 - P| / sqrt(P m + m^2) < 3.8e-6
Each tolerance keeps at least 3.5x margin over the oracle's errors (3.5x on noise, 18x on peak), and each sits below
the defects it must reveal:
    - one lag too many in an E1B row (lag 16368 in the sum) moves the noise by P[16368] / (16368 m) = 6.1e-5 P/m;
    - operands stored at fp16 precision (10-bit mantissa) move peaks by up to 3.7e-4 (C/A) / 3.0e-4 (E1B) and the
      noise by up to 6.4e-5 / 1.4e-5;
    - a profile off by 1e-3 of the row mean at a noise lag is 7e-4 of sqrt(P m + m^2) there.
The engine's own largest errors over test_gpu_precision's cases, on an NVIDIA B200 (1000 W power limit): peak 1.1e-6,
noise 5.0e-7, snr 8.4e-7, profile 4.2e-6."""
import numpy as np

from profile_ref import N, block_lags, code_row, code_spectra64, lags_of, split_dop

PEAK_RTOL = 1e-5
NOISE_RTOL = 2e-5
SNR_RTOL = 3e-5
PROFILE_TAU = 3e-5


class SearchRef:
    """One capture (K blocks in the engine's capture format) of a search with `params` over the table `sats`."""

    def __init__(self, O, params, capture, sats):
        self.O, self.p, self.sats = O, params, sats
        self.K, self.half_bin = int(params.k_noncoh), int(params.half_bin)
        self.bits = int(params.sample_bits) or 1
        self.cap = np.ascontiguousarray(capture, np.uint8).reshape(-1)
        assert self.cap.size == self.K * O.block_bytes(self.bits), (self.cap.size, self.K, self.bits)
        self._D, self._C = {}, {}

    def spectra(self, v):
        """conj(D_b) of the K blocks at half-bin variant v, complex128 [K, N]."""
        if v not in self._D:
            bb = self.O.block_bytes(self.bits)
            x = np.array([self.O.capture_baseband(self.cap[b * bb:(b + 1) * bb], half_rot=v, sample_bits=self.bits)
                          for b in range(self.K)])
            self._D[v] = np.conj(np.fft.fft(x.astype(np.complex128), axis=1))
        return self._D[v]

    def codes(self, sat):
        """(spectrum of row sat, spectrum of the next row), complex128."""
        if sat not in self._C:
            self._C[sat] = code_spectra64(self.O, self.sats, sat)
        return self._C[sat]

    def power(self, sat, h):
        """float64 P over the row's L lags at Doppler index h (half-bins when half_bin)."""
        d, v = split_dop(int(h), self.half_bin)
        C, nxt = self.codes(sat)
        row = code_row(C, nxt, d, self.p.wrap_mode == self.O.WRAP_REFERENCE)
        r = np.fft.ifft(self.spectra(v) * row, axis=1) * N
        L = lags_of(self.sats[sat])
        P = np.zeros(L)
        for b in range(self.K):
            P += np.abs(r[b, block_lags(L, b, int(h), self.K, self.half_bin, self.p.code_doppler)]) ** 2
        return P

    def cells(self, sat, hs=None):
        """(hs, peak, noise, snr, lag, P) over the row's Doppler indices (or hs): Correlate's cell rules on P -- the
        maximum, the mean, their ratio (NaN on a row of zeros) and the first argmax."""
        hs = np.arange(self.p.dop_lo, self.p.dop_hi + 1) if hs is None else np.asarray(hs)
        P = np.array([self.power(sat, h) for h in hs])
        peak, noise = P.max(axis=1), P.mean(axis=1)
        with np.errstate(invalid="ignore"):
            snr = peak / noise
        return hs, peak, noise, snr, P.argmax(axis=1), P


class Worst:
    """The largest errors the checks below have seen: relative for peak / noise / snr, |row - P| / sqrt(P m + m^2) for
    profiles; and how many lags / Dopplers differed inside the tie zone."""

    def __init__(self, label=""):
        self.label = label
        self.peak = self.noise = self.snr = self.profile = 0.0
        self.dop = self.code = self.fine_peak = 0.0   # refinement (refine_ref.check_fine): bins, FS samples, relative
        self.lag_ties = self.dop_ties = 0

    def rel(self, field, got, want):
        e = float(np.max(np.abs(np.asarray(got, np.float64) / want - 1))) if np.size(want) else 0.0
        setattr(self, field, max(getattr(self, field), e))
        return e

    def __str__(self):
        return ("precision [%s]: max rel. error peak %.1e noise %.1e snr %.1e, profile %.1e of sqrt(P m + m^2); "
                "refinement: dop %.1e bin, code_fs %.1e FS samples, peak %.1e; %d lag and %d Doppler ties"
                % (self.label, self.peak, self.noise, self.snr, self.profile, self.dop, self.code, self.fine_peak,
                   self.lag_ties, self.dop_ties))


def check_cells(got, ref, worst, what="", margin=1.0):
    """got: CELL_DTYPE cells of one row at ref's Doppler indices; ref: SearchRef.cells (or CoherentRef.cells).  Peak,
    noise and snr within their tolerances (divided by margin); a lag other than the reference's first argmax only where
    the reference's P there is within PEAK_RTOL of the peak.  Cells whose reference P is all zero (an SBAS row) are
    skipped."""
    hs, peak, noise, snr, lag, P = ref
    got = np.asarray(got).reshape(-1)
    assert got.size == hs.size, (what, got.size, hs.size)
    on = noise > 0
    g = got[on]
    for f, want, tol in (("peak", peak[on], PEAK_RTOL), ("noise", noise[on], NOISE_RTOL), ("snr", snr[on], SNR_RTOL)):
        tol = tol / margin
        e = worst.rel(f, g[f], want)
        assert e <= tol, "%s: %s rel. error %.2e > %.0e at h = %s" % (
            what, f, e, tol, hs[on][np.argmax(np.abs(g[f] / want - 1))])
    L = P.shape[1]
    assert ((g["lag"] >= 0) & (g["lag"] < L)).all(), what
    tie = g["lag"] != lag[on]
    near = P[on][np.arange(g.size), g["lag"]] >= peak[on] * (1 - PEAK_RTOL)
    assert (near | ~tie).all(), "%s: lag off the reference's peak at h = %s" % (what, hs[on][tie & ~near])
    worst.lag_ties += int(tie.sum())


def check_record(rec, ref, worst, what=""):
    """A search record against the row's reference cells: its Doppler the reference's best snr or within SNR_RTOL of
    it, then the cell at that Doppler as check_cells."""
    hs, peak, noise, snr, lag, P = ref
    j = int(rec["dop"]) - int(hs[0])
    assert 0 <= j < hs.size, (what, int(rec["dop"]))
    best = int(np.argmax(snr))
    assert j == best or snr[j] >= snr[best] * (1 - SNR_RTOL), "%s: dop %d (snr %g) vs %d (snr %g)" % (
        what, int(rec["dop"]), snr[j], int(hs[best]), snr[best])
    worst.dop_ties += int(j != best)
    cell = np.array([(rec["peak"], rec["noise"], rec["snr"], rec["lag"])],
                    [("peak", "<f4"), ("noise", "<f4"), ("snr", "<f4"), ("lag", "<i4")])
    check_cells(cell, tuple(a[j:j + 1] for a in ref), worst, what)


def check_profile(row, P, worst, what=""):
    """A lag profile against the reference's P at every lag: |row - P| <= PROFILE_TAU sqrt(P m + m^2)."""
    row = np.asarray(row, np.float64)
    assert row.shape == P.shape, (what, row.shape, P.shape)
    m = P.mean()
    e = np.abs(row - P) / np.sqrt(P * m + m * m)
    worst.profile = max(worst.profile, float(e.max()))
    assert e.max() <= PROFILE_TAU, "%s: profile error %.2e of sqrt(P m + m^2) at lag %d" % (what, e.max(), np.argmax(e))
