"""Float64 reference of the hand-off of coherent records (acq_refine_coherent*, acq_profile_coherent*) and its precision
bound.

Profile.  The profile of a coherent record is CoherentRef.power at the record's index: the coherent search's own P.  Its
peak-quality reduction is profile_ref.peak2_of, and search_ref.check_profile's bound applies to the rows.

Refinement.  CoherentHandoffRef evaluates k_refine_coh's five correlations in every block b = g M + j of a record (h, n):
(h - H, n), (h, n - 1), (h, n), (h, n + 1), (h + H, n), H = 1 + half_bin, each Doppler point at its own code row and
spectrum variant (d', v') = split_h(h +- H, F), at lag n_b = n + 16 b of block b's inverse FFT (profile_ref.block_lags).
Block j of a group enters each point's group sum rotated by coherent_ref.theta(j, d', v'), and every group takes the
data-bit hypothesis that is the first maximum at the centre (h, n) -- "no edge", then s = 1..M-1 -- for all five sums.
A code row d' puts e^{+j 2 pi d' n_b / N} on block b's sum; theta_j removes its 16 j d' part, so what is left on a group
sum is the phase of the group's first block, n_b0 = n + 16 g M, and the outer points are multiplied by
e^{-j 2 pi (d' - d) n_b0 / N} (corr = -1; corr = +1 is the wrong sign, for the tests that pin it).  Then
refine_ref.combine's estimator over the groups: delta and eps from num / den and early / late, dop_hz = (h + H delta)
BIN / F, code_fs = 4 (n + eps), peak = sum over the groups of |X_g(h, n)|^2.  At M = 1 this is RefineRef.fine.

Error model.  Each fp32 block sum of k_refine_coh carries refine_ref's REFINE_TAU sqrt(m_b) (m_b: the block's mean lag
power in that code row and variant); the rotation by theta_j (sincospif, one complex fma) and the signed prefix sums add a
few ulp of |u_j|.  So a group sum is off by at most c_s sum_j (REFINE_TAU sqrt(m_j) + 8 u |u_j|), c_s = 1 for "no edge"
and 3 for 2 S_s - T.  These per-point errors go through num / den and early / late to first order as in
refine_ref.combine, with the fp32 sums over the G groups.  A group whose two best hypotheses at the centre lie within
HYP_RTOL of each other may be signed either way by fp32 arithmetic: the reference then also offers the other choice."""
import numpy as np

from coherent_ref import CoherentRef, split_h, theta
from profile_ref import N, code_row
from refine_ref import BIN_HZ, DECIM, REFINE_TAU, U32, _clamp, _f32, _ratio_bound

LAGS_L1 = 4092
HYP_RTOL = 1e-4
POINT = [0, 1, 1, 1, 2]   # Doppler point (h - H, h, h + H) of each of the five sums
DLAG = [0, -1, 0, 1, 0]   # lag offset of each of the five sums


class CoherentHandoffRef(CoherentRef):
    """CoherentRef of one capture and satellite, with the refinement of coherent records."""

    def row(self, b, d, v, F):
        """r_b over all N lags of its inverse FFT at code row d and spectrum variant v (complex128)."""
        key = ("row", b, d, v, F)
        if key not in self._D:
            code = code_row(self.C, self.nxt, d, self.p.wrap_mode == self.O.WRAP_REFERENCE)
            self._D[key] = np.fft.ifft(np.conj(self.spectrum(b, v, F)) * code) * N
        return self._D[key]

    def blocks(self, h, n, m_coh, sign16=-1):
        """(U [G, M, 5] complex128: the rotated block sums u_j of the five points; m [G, M, 5]: their blocks' mean lag
        power; dd [3]: code row of each Doppler point)."""
        M = int(m_coh)
        H = 1 + int(self.p.half_bin)
        F = M * H
        pts = [split_h(int(h) + (i - 1) * H, F) for i in range(3)]
        G = self.K // M
        U = np.zeros((G, M, 5), np.complex128)
        m = np.zeros((G, M, 5))
        for g in range(G):
            for j in range(M):
                b = g * M + j
                nb = (int(n) + 16 * b) % N if self.K > 1 else int(n)
                for i, (d, v) in enumerate(pts):
                    r = self.row(b, d, v, F)
                    rot = np.exp(1j * theta(j, d, v, F, sign16))
                    for p in range(5):
                        if POINT[p] == i:
                            U[g, j, p] = rot * r[(nb + DLAG[p]) % N]
                            m[g, j, p] = np.mean(np.abs(r) ** 2)
        return U, m, [d for d, _ in pts]

    def fine(self, h, n, m_coh, tau=REFINE_TAU, corr=-1, sign16=-1):
        """The refinement of a record at (h, n): a list of dicts of float64 scalars (delta, eps, bounds, dop_hz, code_fs,
        peak) -- the first for the reference's hypotheses, the others for the near-tie alternatives."""
        M = int(m_coh)
        U, m, dd = self.blocks(h, n, M, sign16)
        G = U.shape[0]
        T = U.sum(axis=1)                                                    # [G, 5]
        S = np.stack([U[:, :s].sum(axis=1) for s in range(1, M)], axis=1) if M > 1 else np.zeros((G, 0, 5))
        hyp = np.concatenate([np.abs(T[:, None, 2]) ** 2, np.abs(2 * S[:, :, 2] - T[:, None, 2]) ** 2], axis=1)
        choice = np.argmax(hyp, axis=1)                                      # first maximum
        alts = [choice]
        for g in range(G):
            order = np.argsort(-hyp[g], kind="stable")
            if M > 1 and hyp[g, order[1]] >= hyp[g, order[0]] * (1 - HYP_RTOL):
                c2 = choice.copy()
                c2[g] = order[1]
                alts.append(c2)
        eb = tau * np.sqrt(m) + 8 * U32 * np.abs(U)                           # per block and point
        out = []
        for ch in alts:
            X = np.where(ch[:, None] == 0, T, 0)
            for g in range(G):
                if ch[g]:
                    X[g] = 2 * S[g, ch[g] - 1] - T[g]
            e = eb.sum(axis=1) * np.where(ch > 0, 3.0, 1.0)[:, None]
            nb0 = (int(n) + 16 * M * np.arange(G)) % N
            for p, i in ((0, 0), (4, 2)):
                X[:, p] = X[:, p] * np.exp(corr * 2j * np.pi * (dd[i] - dd[1]) * nb0 / N)
            out.append(combine_groups(X, e, int(h), int(n), M, 1 + int(self.p.half_bin)))
        return out


def combine_groups(X, e, h, n, M, H):
    """refine_ref.combine's estimator over the group sums X [G, 5] (phase-corrected) with per-sum errors e [G, 5]."""
    G = X.shape[0]
    Xm, X0, Xp = X[:, 0], X[:, 2], X[:, 4]
    a, g = Xm - Xp, 2 * X0 - Xm - Xp
    num, den = np.sum((a * np.conj(g)).real), np.sum(np.abs(g) ** 2)
    early, late = np.sum((X[:, 1] * np.conj(X0)).real), np.sum((X[:, 3] * np.conj(X0)).real)
    peak = np.sum(np.abs(X0) ** 2)
    gam = (G + 4) * U32
    ea, eg = e[:, 0] + e[:, 4], 2 * e[:, 2] + e[:, 0] + e[:, 4]
    dnum = np.sum(ea * np.abs(g) + np.abs(a) * eg + ea * eg) + gam * np.sum(np.abs(a) * np.abs(g))
    dden = np.sum(2 * np.abs(g) * eg + eg * eg) + gam * den
    A1, A2, A3 = np.abs(X[:, 1]), np.abs(X0), np.abs(X[:, 3])
    de = np.sum(e[:, 1] * A2 + A1 * e[:, 2] + e[:, 1] * e[:, 2]) + gam * np.sum(A1 * A2)
    dl = np.sum(e[:, 3] * A2 + A3 * e[:, 2] + e[:, 3] * e[:, 2]) + gam * np.sum(A3 * A2)
    delta = num / den if den > 0 else 0.0
    eps = 3.0 * (late - early) / (early + late) if early + late > 0 else 0.0
    F = M * H
    return dict(h=h, n=n, M=M, F=F, delta=delta, eps=eps,
                b_delta=_ratio_bound(num, den, dnum, dden) + 2 * U32,
                b_eps=3.0 * _ratio_bound(late - early, early + late, de + dl, de + dl) + 2 * U32,
                dop_hz=(h + H * _clamp(delta)) * BIN_HZ / F, code_fs=DECIM * (n + _clamp(eps)),
                peak=peak, b_peak=np.sum(2 * A2 * e[:, 2] + e[:, 2] ** 2) + gam * peak)


def _ulp(x):
    return float(np.spacing(np.float32(abs(x))))


def expected(f):
    """dop_hz [lo, hi], code_fs [lo, hi] and the ca_shift set of an fp32 refinement within f's bounds: the delta / eps
    intervals (clamped) through k_refine_coh's output arithmetic, (fl(h / F) + fl(delta / M)) BIN, widened by its
    roundings, and refine_ref.expected's code_fs rule."""
    dlo, dhi = _clamp(f["delta"] - f["b_delta"]), _clamp(f["delta"] + f["b_delta"])
    elo, ehi = _clamp(f["eps"] - f["b_eps"]), _clamp(f["eps"] + f["b_eps"])
    c = f["h"] / f["F"]
    hz = [(c + x / f["M"]) * BIN_HZ for x in (dlo, dhi)]
    slack = 2 * (_ulp(c) + _ulp(1.0)) * BIN_HZ + 2 * max(_ulp(hz[0]), _ulp(hz[1]))
    fs = [DECIM * _f32(f["n"] + x) for x in (elo, ehi)]
    shifts = {s % (DECIM * LAGS_L1) for s in range(int(np.rint(fs[0])), int(np.rint(fs[1])) + 1)}
    return [hz[0] - slack, hz[1] + slack], fs, shifts


def check_fine_coherent(fine, rec, refs, m_coh, worst, what="", peak_rtol=1e-5):
    """acq_fine rows of coherent records against the reference: dop_hz and code_fs inside the bound of one of the
    reference's hypothesis choices, ca_shift in its set, peak within max(peak_rtol, the model's bound).  refs: sat ->
    CoherentHandoffRef of the record's capture."""
    fine, rec = np.asarray(fine).reshape(-1), np.asarray(rec).reshape(-1)
    assert fine.size == rec.size, (what, fine.size, rec.size)
    for i, (g, r) in enumerate(zip(fine, rec)):
        w = "%s record %d (sat %d dop %d lag %d)" % (what, i, r["sat"], r["dop"], r["lag"])
        cands = refs(i, r).fine(int(r["dop"]), int(r["lag"]), m_coh)
        errs = []
        for f in cands:
            (hlo, hhi), (clo, chi), shifts = expected(f)
            tol = max(peak_rtol * f["peak"], f["b_peak"])
            ok = (hlo <= g["dop_hz"] <= hhi and clo <= g["code_fs"] <= chi and int(g["ca_shift"]) in shifts
                  and abs(float(g["peak"]) - f["peak"]) <= tol)
            errs.append("dop_hz %.9g in [%.9g, %.9g]? code_fs %.9g in [%.9g, %.9g]? ca_shift %d in %s? peak %.7g vs %.7g "
                        "(tol %.1e)" % (g["dop_hz"], hlo, hhi, g["code_fs"], clo, chi, g["ca_shift"], sorted(shifts),
                                        g["peak"], f["peak"], tol))
            if ok:
                worst.dop = max(worst.dop, abs(float(g["dop_hz"]) - f["dop_hz"]) / BIN_HZ)
                worst.code = max(worst.code, abs(float(g["code_fs"]) - f["code_fs"]))
                worst.fine_peak = max(worst.fine_peak, abs(float(g["peak"]) / f["peak"] - 1) if f["peak"] else 0.0)
                break
        else:
            raise AssertionError("%s: %s" % (w, "; ".join(errs)))
