"""Float64 reference of the hand-off refinement (acq_refine, acq_refine_device: k_refine) and its precision bound.

RefineRef evaluates, on SearchRef's float64 spectra, the five correlations k_refine sums around a record (dop h, lag n)
in each block b: r_{d-1}[n_b], r_d[n_b - 1], r_d[n_b], r_d[n_b + 1] and r_{d+1}[n_b], with d the whole bin of h (so on
half-bins the neighbours are +-1 whole bin at h's variant), n_b = (n + 16 b + s(b, h)) mod N the lag of the undelayed
block (profile_ref.block_lags; s = 0 without code_doppler), and the code rows and wraps of profile_ref.code_row.  One
inverse FFT per (block, code row) gives all five.  It then applies orc_refine's combine in float64: the X-/X+ phases
e^{+-j 2 pi n_b / N}, num, den, early, late and peak summed over the blocks, the +-1 clamps, the slopes 3 (C/A) and 1/3
(E1B), dop_hz, code_fs and ca_shift.

Error model.  k_refine forms each of the five values as a direct fp32 sum of 16384 products of fp32 spectra, fp32 code
rows and fp32 twiddles, so each carries an absolute error of about REFINE_TAU sqrt(m_b), m_b the block's mean lag power
(over all N lags) in that code row.  Carried to first order through num / den and early / late -- with the reference's
own float64 magnitudes, plus the fp32 rounding of the K-block sums of the combine -- that gives a bound on |d delta| and
|d eps| per record; a ratio num / den whose den the perturbation could reach is unbounded, and the check then accepts
anything the clamp allows.  The fp32 outputs add their own floor: code_fs = 4 (float)(n + eps) cannot resolve eps
better than ulp(n) (9.8e-4 FS samples for C/A lags, 3.9e-3 above lag 8192), dop_hz = (c + delta) BIN with c the
record's centre in bins rounds at ulp(c) (2.4e-4 bin at 2048 bins) and ulp(dop_hz) (0.031 Hz there), both about 2e-6 bin
at 20 bins.  peak is held to PEAK_RTOL of the reference's sum of |r_d[n_b]|^2, or to the model's bound where that is
looser (a placed record at a lag of little power).

REFINE_TAU is pinned by a numpy fp32 emulation of k_refine in its summation order (tests/test_refine_ref_cpu.py) on
the oracle's fp32 spectra: over its seven shapes the largest |R32 - R| / sqrt(m_b) is 1.27e-6, so REFINE_TAU = 4e-6
keeps a 3.1x margin; the emulation's delta and eps stay far inside the bound built on REFINE_TAU / 3 (largest errors
7e-8 bin, 3e-7).  The same emulation with the block phase missing its code-Doppler shift, or its 16 b advance, fails.
The engine's largest errors against this reference over test_gpu_precision's refinements (records of every search
kernel and 25 placements of records at the range's edges, lags 0 and L - 1 and noise rows), on an NVIDIA B200 (1000 W
power limit): dop 4.9e-6 bin, code_fs 1.9e-3 FS samples (the ulp of code_fs), peak 2.2e-6 (6.2e-7 at search
records); over test_gpu_limits' (+-2048 bins, K = 255, 33 code-Doppler copies): dop 8.0e-5 bin, where dop_hz's own
ulp is 0.031 Hz = 1.2e-4 bin."""
import numpy as np

from profile_ref import LAGS_E1B, LAGS_L1, N, code_row, code_shift, lags_of, split_dop
from search_ref import PEAK_RTOL, SearchRef

BIN_HZ = 16.368e6 / 65536
DECIM = 4
REFINE_TAU = 4e-6
U32 = 2.0 ** -24


class RefineRef(SearchRef):
    """SearchRef of one capture, with the refinement of records at any (sat, dop, lag) the engine accepts."""

    def points(self, sat, h, n):
        """(R [K, 5] complex128: r_{d-1}[n_b], r_d[n_b - 1], r_d[n_b], r_d[n_b + 1], r_{d+1}[n_b]; m [K, 3]: mean lag
        power of rows d - 1, d, d + 1; n_b [K])."""
        d, v = split_dop(int(h), self.half_bin)
        C, nxt = self.codes(sat)
        ref_wrap = self.p.wrap_mode == self.O.WRAP_REFERENCE
        D = self.spectra(v)
        r = [np.fft.ifft(D * code_row(C, nxt, d + j, ref_wrap), axis=1) * N for j in (-1, 0, 1)]
        b = np.arange(self.K)
        shift = np.array([code_shift(i, int(h), self.half_bin) for i in b]) if self.p.code_doppler else 0
        nb = (int(n) + 16 * b + shift) % N
        R = np.stack([r[0][b, nb], r[1][b, (nb - 1) % N], r[1][b, nb], r[1][b, (nb + 1) % N], r[2][b, nb]], axis=1)
        m = np.stack([np.mean(np.abs(x) ** 2, axis=1) for x in r], axis=1)
        return R, m, nb

    def fine(self, sat, h, n, tau=REFINE_TAU):
        """The refinement of a record at (sat, dop h, lag n) with its bounds: a dict of float64 scalars."""
        return combine(*self.points(sat, h, n), h=int(h), n=int(n), half_bin=self.half_bin,
                       e1b=lags_of(self.sats[sat]) == LAGS_E1B, tau=tau)


def _ratio_bound(num, den, dnum, dden):
    """Bound on |(num + x) / (den + y) - num / den| for |x| <= dnum, |y| <= dden (inf where den + y may reach 0)."""
    if den - dden <= 0:
        return np.inf
    return (dnum + abs(num / den) * dden) / (den - dden)


def combine(R, m, nb, h, n, half_bin, e1b, tau=REFINE_TAU):
    """orc_refine's combine of the five points per block in float64, and the error bounds of the fp32 kernel's."""
    K = R.shape[0]
    w = np.exp(2j * np.pi * nb / N)
    Xm, Xp, X0 = R[:, 0] * w, R[:, 4] * np.conj(w), R[:, 2]
    a, g = Xm - Xp, 2 * X0 - Xm - Xp
    num, den = np.sum((a * np.conj(g)).real), np.sum(np.abs(g) ** 2)
    early, late = np.sum((R[:, 1] * np.conj(R[:, 2])).real), np.sum((R[:, 3] * np.conj(R[:, 2])).real)
    peak = np.sum(np.abs(R[:, 2]) ** 2)
    # per-point absolute error of the fp32 sums (rows d - 1, d, d, d, d + 1)
    e = tau * np.sqrt(m[:, [0, 1, 1, 1, 2]])
    gam = (K + 4) * U32   # the fp32 K-block sums and products of the combine
    ea, eg = e[:, 0] + e[:, 4], 2 * e[:, 2] + e[:, 0] + e[:, 4]
    dnum = np.sum(ea * np.abs(g) + np.abs(a) * eg + ea * eg) + gam * np.sum(np.abs(a) * np.abs(g))
    dden = np.sum(2 * np.abs(g) * eg + eg * eg) + gam * den
    A1, A2, A3 = np.abs(R[:, 1]), np.abs(R[:, 2]), np.abs(R[:, 3])
    de = np.sum(e[:, 1] * A2 + A1 * e[:, 2] + e[:, 1] * e[:, 2]) + gam * np.sum(A1 * A2)
    dl = np.sum(e[:, 3] * A2 + A3 * e[:, 2] + e[:, 3] * e[:, 2]) + gam * np.sum(A3 * A2)
    slope = 1.0 / 3.0 if e1b else 3.0
    delta = num / den if den > 0 else 0.0
    eps = slope * (late - early) / (early + late) if early + late > 0 else 0.0
    b_delta = _ratio_bound(num, den, dnum, dden) + 2 * U32
    b_eps = slope * _ratio_bound(late - early, early + late, de + dl, de + dl) + 2 * U32
    c = 0.5 * h if half_bin else float(h)
    return dict(c=c, n=n, L=LAGS_E1B if e1b else LAGS_L1, delta=delta, eps=eps, b_delta=b_delta, b_eps=b_eps,
                peak=peak, b_peak=np.sum(2 * A2 * e[:, 2] + e[:, 2] ** 2) + gam * peak)


def _clamp(x):
    return min(1.0, max(-1.0, x))


def _f32(x):
    return float(np.float32(x))


def intervals(f):
    """([lo, hi] of delta, [lo, hi] of eps): the reference's values within their bounds, through the +-1 clamps."""
    return ([_clamp(f["delta"] - f["b_delta"]), _clamp(f["delta"] + f["b_delta"])],
            [_clamp(f["eps"] - f["b_eps"]), _clamp(f["eps"] + f["b_eps"])])


def expected(f):
    """The intervals the fp32 outputs of a refinement within the bound fall in: dop_hz [lo, hi] and code_fs [lo, hi] --
    the delta / eps intervals through the output roundings (monotone, so the ends map to the ends): k_refine's
    ((float)c + delta) * (float)BIN, c and BIN exact in fp32, or orc_refine's one rounding of the double product -- and
    the set of ca_shift = lrint(code_fs) mod 4 L over the code_fs interval."""
    d, e = intervals(f)
    hz = [(min if i == 0 else max)(_f32(_f32(f["c"] + x) * BIN_HZ), _f32((f["c"] + x) * BIN_HZ)) for i, x in enumerate(d)]
    fs = [DECIM * _f32(f["n"] + x) for x in e]   # 4 * ((float)n + eps); orc_refine's (float)(4 (n + eps)) is the same
    shifts = {s % (DECIM * f["L"]) for s in range(int(np.rint(fs[0])), int(np.rint(fs[1])) + 1)}
    return hz, fs, shifts


def check_fine(fine, rec, ref, worst, what="", margin=1.0):
    """acq_fine rows against the reference's refinement of the same records (acq_record rows): dop_hz and code_fs inside
    the bound of the reference's delta / eps (clamped, plus the fp32 output floor), ca_shift the reference's (either
    side where the code_fs interval straddles a half-integer), peak within PEAK_RTOL (or the model's bound where looser).
    margin > 1 divides REFINE_TAU and PEAK_RTOL by it (the fp32 outputs' floors stay)."""
    fine, rec = np.asarray(fine).reshape(-1), np.asarray(rec).reshape(-1)
    assert fine.size == rec.size, (what, fine.size, rec.size)
    for i, (g, r) in enumerate(zip(fine, rec)):
        f = ref.fine(int(r["sat"]), int(r["dop"]), int(r["lag"]), tau=REFINE_TAU / margin)
        w = "%s record %d (sat %d dop %d lag %d)" % (what, i, r["sat"], r["dop"], r["lag"])
        (hlo, hhi), (clo, chi), shifts = expected(f)
        got_d = float(g["dop_hz"]) / BIN_HZ
        worst.dop = max(worst.dop, abs(got_d - (f["c"] + _clamp(f["delta"]))))
        worst.code = max(worst.code, abs(float(g["code_fs"]) - DECIM * (f["n"] + _clamp(f["eps"]))))
        assert hlo <= g["dop_hz"] <= hhi, "%s: dop_hz %.9g outside [%.9g, %.9g] (delta %.9f, bound %.2e bin)" % (
            w, g["dop_hz"], hlo, hhi, f["delta"], f["b_delta"])
        assert clo <= g["code_fs"] <= chi, "%s: code_fs %.9g outside [%.9g, %.9g] (eps %.9f, bound %.2e)" % (
            w, g["code_fs"], clo, chi, f["eps"], f["b_eps"])
        assert int(g["ca_shift"]) in shifts, (w, int(g["ca_shift"]), shifts)
        tol = max(PEAK_RTOL / margin * f["peak"], f["b_peak"])
        worst.fine_peak = max(worst.fine_peak, abs(float(g["peak"]) / f["peak"] - 1))
        assert abs(float(g["peak"]) - f["peak"]) <= tol, "%s: peak %.7g vs %.7g (tol %.2e)" % (w, g["peak"], f["peak"], tol)
