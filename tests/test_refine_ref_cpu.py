"""CPU side of the refinement's precision bound (tests/refine_ref.py): the oracle's refinement (double sums over its fp32
spectra) and a numpy fp32 emulation of k_refine in its summation order against the float64 RefineRef.  The emulation
passing with a 3x margin on REFINE_TAU shows that fp32 arithmetic meets the bound the GPU tests hold k_refine to; the
same emulation with the block phase of the X-/X+ points missing its code-Doppler shift, or its 16 b block advance, must
not pass."""
import numpy as np
import pytest

from flydog_sdr_gps_b200 import engine, synth
from flydog_sdr_gps_b200 import sats as S

from profile_ref import N, code_row, code_shift, lags_of, split_dop
from refine_ref import BIN_HZ, DECIM, REFINE_TAU, RefineRef, check_fine, intervals
from search_ref import Worst

BIN = engine.BIN_HZ

CASES = {
    # (table, params, signals, sel, sample_bits, code-Doppler capture): test_oracle_cpu's refinement shapes and the
    # formats and wraps of test_search_ref_cpu
    "ca_k1": ("ref", dict(), [(2, 4001, 3.3 * BIN, 50, 1.0), (10, 12346, -7.45 * BIN, 48, 2.0)], [2, 10, 20], 1, False),
    "ca_k4_half_bins": ("nav", dict(k_noncoh=4, half_bin=1, dop_lo=-20, dop_hi=20),
                        [(7, 8002, 4.5 * BIN, 46, 0.5), (12, 100, -3.1 * BIN, 46, 0.1)], [7, 12], 1, False),
    # s(b, h) = round(b h / 385) reaches -2 in block 5 at h = -160: shifted and unshifted blocks in one record
    "ca_k6_code_doppler": ("nav", dict(k_noncoh=6, code_doppler=1, dop_lo=-166, dop_hi=-154),
                           [(8, 640, -160.3 * BIN, 45, 2.0)], [8, 3], 1, True),
    "e1b_k1": ("e1b", dict(dop_lo=-8, dop_hi=8), [(1, 30003, -6.2 * BIN, 50, 0.4)], [1, 4], 1, False),
    "e1b_k4": ("e1b", dict(k_noncoh=4, dop_lo=-3, dop_hi=3), [(1, 30000, -2.3 * BIN, 44, 0.4)], [1, 2], 1, False),
    "ca_2bit": ("nav", dict(sample_bits=2), [(12, 333, -3.4 * BIN, 47, 0.7)], [12, 13], 2, False),
    # row 30's negative bins read row 31 in the reference wrap; here its own row
    "ca_k3_circular_wrap": ("nav", dict(k_noncoh=3, wrap_mode=1), [(30, 700, -8.3 * BIN, 46, 0.3)], [30, 31], 1, False),
}


def _case(O, name):
    which, kw, sig, sel, bits, cd = CASES[name]
    table = {"ref": S.reference_table, "nav": S.navstar, "e1b": lambda: S.e1b(range(1, 6))}[which]()
    K = kw.get("k_noncoh", 1)
    cap = synth.make_capture(29, K, table, sig, sample_bits=bits, code_doppler=cd)
    p = O.default_params(**kw)
    rec = O.search(cap, table, sel=sel, params=p)
    return table, p, cap, rec


# ---------------------------------------------------------------- fp32 emulation of k_refine
def _cmul(ax, ay, bx, by):
    return ax * bx - ay * by, ax * by + ay * bx


def _tw(k):
    """fp32 e^{+j pi k / 8192} of integer k (sincospif of an exact argument)."""
    a = np.pi * np.asarray(k, np.float64) / 8192.0
    return np.cos(a).astype(np.float32), np.sin(a).astype(np.float32)


# thread t sums k = 4 (t + 256 i) + k2 for k2 = 0..3 (outer), i = 0..15 (inner)
_ORDER = np.array([[4 * (t + 256 * i) + k2 for t in range(256)] for k2 in range(4) for i in range(16)])


def _cta_sum(x):
    """k_refine's reduction of 16384 fp32 terms: per-thread sequential sums in _ORDER, a 32-lane xor tree, 8 warps in
    order."""
    acc = np.zeros(256, np.float32)
    for s in range(_ORDER.shape[0]):
        acc = acc + x[_ORDER[s]]
    a = acc.reshape(8, 32)
    for off in (16, 8, 4, 2, 1):
        a = a[:, :off] + a[:, off:2 * off]
    r = np.float32(0)
    for w in range(8):
        r = r + a[w, 0]
    return r


def emulate_k_refine(O, p, cap, sats, rec, phase="n + 16 b + cshift"):
    """(FINE_DTYPE rows, fp32 (delta, eps) before the output roundings [n, 2], the five fp32 sums of every block
    [n, K, 5] as complex128) of k_refine on fp32 spectra (the oracle's
    fp32 FFTs of the delayed blocks and of the code basebands), fp32 products and twiddles, in the kernel's summation
    order.  phase: the block phase of X-/X+, the kernel's or one with a term missing ("n + 16 b", "n + cshift")."""
    K, hb, bits = int(p.k_noncoh), int(p.half_bin), int(p.sample_bits) or 1
    bb = O.block_bytes(bits)
    cap = np.ascontiguousarray(cap, np.uint8).reshape(-1)
    k = np.arange(N)
    out = np.zeros(len(rec), O.FINE_DTYPE)
    inner = np.zeros((len(rec), 2))
    sums = np.zeros((len(rec), int(p.k_noncoh), 5), np.complex128)
    for i, r in enumerate(rec):
        sat, h, n = int(r["sat"]), int(r["dop"]), int(r["lag"])
        e1b = lags_of(sats[sat]) != 4092
        d, v = split_dop(h, hb)
        C = O.code_spectrum(sats[sat])
        nxt = O.code_spectrum(sats[sat + 1]) if sat + 1 < len(sats) else np.zeros(N, np.complex64)
        E = [code_row(C, nxt, d + j, p.wrap_mode == O.WRAP_REFERENCE) for j in (-1, 0, 1)]
        w0x, w0y = _tw((k * n) & (N - 1))
        wkx, wky = _tw(k)
        num = den = early = late = peak = np.float32(0)
        for b in range(K):
            cs = code_shift(b, h, hb) if p.code_doppler else 0
            x = O.capture_baseband(cap[b * bb:(b + 1) * bb], half_rot=v, sample_bits=bits)
            D = O.fft16384(np.roll(x, 16 * b + cs), -1)   # the front end's circular delay of block b
            terms = []
            for j in range(3):   # conj(d) * E[k - dd] * w0
                px = D.real * E[j].real + D.imag * E[j].imag
                py = D.real * E[j].imag - D.imag * E[j].real
                terms.append(_cmul(px, py, w0x, w0y))
            pc = terms[1]
            pts = [terms[0], _cmul(*pc, wkx, -wky), pc, _cmul(*pc, wkx, wky), terms[2]]
            R = [(_cta_sum(tx), _cta_sum(ty)) for tx, ty in pts]
            sums[i, b] = [complex(x, y) for x, y in R]
            lag = {"n + 16 b + cshift": n + 16 * b + cs, "n + 16 b": n + 16 * b, "n + cshift": n + cs}[phase]
            cx, sy = _tw(lag & (N - 1))
            Xm = _cmul(*R[0], cx, sy)
            Xp = _cmul(*R[4], cx, -sy)
            X0 = R[2]
            a = (Xm[0] - Xp[0], Xm[1] - Xp[1])
            g = ((X0[0] + X0[0]) - Xm[0] - Xp[0], (X0[1] + X0[1]) - Xm[1] - Xp[1])
            num = num + (a[0] * g[0] + a[1] * g[1])
            den = den + (g[0] * g[0] + g[1] * g[1])
            early = early + (R[1][0] * R[2][0] + R[1][1] * R[2][1])
            late = late + (R[3][0] * R[2][0] + R[3][1] * R[2][1])
            peak = peak + (R[2][0] * R[2][0] + R[2][1] * R[2][1])
        delta = np.clip(num / den if den > 0 else np.float32(0), -1, 1).astype(np.float32)
        slope = np.float32(1.0 / 3.0) if e1b else np.float32(3.0)
        eps = np.clip(slope * (late - early) / (early + late) if early + late > 0 else np.float32(0), -1, 1)
        eps = np.float32(eps)
        centre = np.float32(0.5) * np.float32(h) if hb else np.float32(h)
        out[i]["dop_hz"] = (centre + delta) * np.float32(BIN_HZ)
        out[i]["code_fs"] = np.float32(DECIM) * (np.float32(n) + eps)
        out[i]["peak"] = peak
        out[i]["ca_shift"] = int(np.rint(out[i]["code_fs"])) % (DECIM * lags_of(sats[sat]))
        inner[i] = delta, eps
    return out, inner, sums


@pytest.mark.parametrize("name", sorted(CASES))
def test_oracle_refine_within_the_bound(oracle, name):
    """orc_refine (double sums over the oracle's fp32 spectra) against the float64 reference: within the bound."""
    table, p, cap, rec = _case(oracle, name)
    worst = Worst("oracle refine " + name)
    check_fine(oracle.refine(cap, table, rec, params=p), rec, RefineRef(oracle, p, cap, table), worst, name)
    print(worst)


@pytest.mark.parametrize("name", sorted(CASES))
def test_fp32_emulation_within_a_third_of_the_bound(oracle, name):
    """k_refine's arithmetic in fp32: every one of the five sums of every block within REFINE_TAU / 3 sqrt(m_b) of the
    reference's, its delta and eps within the bound built on REFINE_TAU / 3, and its outputs within that bound (and
    PEAK_RTOL / 3) through the output roundings."""
    table, p, cap, rec = _case(oracle, name)
    ref = RefineRef(oracle, p, cap, table)
    out, inner, sums = emulate_k_refine(oracle, p, cap, table, rec)
    worst = Worst("fp32 refine " + name)
    tau = 0.0
    for i, r in enumerate(rec):
        R, m, _ = ref.points(int(r["sat"]), int(r["dop"]), int(r["lag"]))
        tau = max(tau, float(np.max(np.abs(sums[i] - R) / np.sqrt(m[:, [0, 1, 1, 1, 2]]))))
        (dlo, dhi), (elo, ehi) = intervals(ref.fine(int(r["sat"]), int(r["dop"]), int(r["lag"]), tau=REFINE_TAU / 3))
        assert dlo <= inner[i, 0] <= dhi and elo <= inner[i, 1] <= ehi, (name, i, inner[i], (dlo, dhi), (elo, ehi))
    print("%s: largest |R32 - R| / sqrt(m) %.2e (REFINE_TAU %.0e)" % (name, tau, REFINE_TAU))
    assert tau <= REFINE_TAU / 3, tau
    check_fine(out, rec, ref, worst, name, margin=3.0)
    print(worst)


@pytest.mark.parametrize("name,phase", [("ca_k6_code_doppler", "n + 16 b"), ("ca_k6_code_doppler", "n + cshift"),
                                        ("ca_k4_half_bins", "n + cshift")])
def test_block_phase_without_a_term_fails(oracle, name, phase):
    """The X-/X+ block phase without its code-Doppler shift, or without its 16 b advance, moves dop_hz outside the bound."""
    table, p, cap, rec = _case(oracle, name)
    with pytest.raises(AssertionError, match="dop_hz"):
        check_fine(emulate_k_refine(oracle, p, cap, table, rec, phase)[0], rec, RefineRef(oracle, p, cap, table),
                   Worst(), name)
