"""Reference side of the peak-quality tests (acq_profile): the power vector that the oracle's Correlate restatement
(oracle/acq_oracle.c, correlate_one) forms at one Doppler index, summed over the K blocks, rebuilt from the oracle's own
exported stages -- capture baseband, code spectrum, 16384-point FFT -- with nothing new but the indexing; and the
second-peak reduction over such a vector.  The indexing helpers (code_row, block_lags) are the one statement of
correlate_one's addressing that the float64 references (search_ref, coherent_ref) use too."""
import numpy as np

N = 16384
LAGS_L1, LAGS_E1B = 4092, 16368
E1B = 3


def code_shift(b, h, half_bin):
    """orc_code_shift: s(b, h) = round-half-away(b h / (385 hb)) in exact integers."""
    d = 385 * (2 if half_bin else 1)
    a = b * h
    s = (2 * abs(a) + d) // (2 * d)
    return -s if a < 0 else s


def lags_of(sat):
    """L of a table row (prn, t1, t2, type): 16368 lags for E1B, 4092 otherwise."""
    return LAGS_E1B if sat[3] == E1B else LAGS_L1


def code_spectra64(O, sats, sat):
    """complex128 spectra of row sat and of the next row (zeros after the last row): float64 FFTs of the oracle's code
    baseband (the decimated +-1 chips; zeros for an SBAS row)."""
    def fft(s):
        return np.fft.fft(O.code_baseband(sats[s]).astype(np.complex128)) if s < len(sats) else np.zeros(N, np.complex128)
    return fft(sat), fft(sat + 1)


def split_dop(dop, half_bin):
    """(d, v) of Doppler index dop: the integer bin d and the half-bin variant v (0 on full bins)."""
    v = (dop & 1) if half_bin else 0
    return ((dop - v) // 2 if half_bin else dop), v


def code_row(C, nxt, d, reference_wrap):
    """correlate_one's code row for bin d, code[(k - d) mod N], in C's dtype: for a negative d the bins past the end of
    the doubled row come from the next table row's spectrum nxt (reference wrap; zeros after the last row) or from the
    same row (circular wrap)."""
    j = np.arange(N) - d
    code = C[j % N].copy()
    past = j >= N   # only for d < 0
    if reference_wrap:
        code[past] = nxt[j[past] - N]
    return code


def block_lags(L, b, dop, K, half_bin, code_doppler):
    """Where lag n of the search sits in block b's IFFT: (n + 16 b + s(b, dop)) mod N for K > 1 (s = 0 without
    code_doppler), n for K = 1."""
    n = np.arange(L)
    if K == 1:
        return n
    return (n + 16 * b + (code_shift(b, dop, half_bin) if code_doppler else 0)) % N


def orc_profile(O, params, capture, sats, sat, dop):
    """float64 [L]: sum over the K blocks of |r_b[block_lags]|^2, r_b = IFFT(conj(D_b) * code_row(d)), from the oracle's
    fp32 spectra and fp32 FFTs.  dop is the Doppler index (half-bins when half_bin)."""
    K, half_bin = int(params.k_noncoh), int(params.half_bin)
    bits = int(params.sample_bits) or 1
    bb = O.block_bytes(bits)
    d, v = split_dop(dop, half_bin)
    C = O.code_spectrum(sats[sat])
    nxt = O.code_spectrum(sats[sat + 1]) if sat + 1 < len(sats) else np.zeros(N, np.complex64)
    code = code_row(C, nxt, d, params.wrap_mode == O.WRAP_REFERENCE)
    L = lags_of(sats[sat])
    cap = np.ascontiguousarray(capture, np.uint8).reshape(-1)
    P = np.zeros(L, np.float64)
    for b in range(K):
        D = O.fft16384(O.capture_baseband(cap[b * bb:(b + 1) * bb], half_rot=v, sample_bits=bits), -1)
        r = O.fft16384(np.conj(D) * code, +1).astype(np.complex128)
        P += np.abs(r[block_lags(L, b, dop, K, half_bin, params.code_doppler)]) ** 2
    return P


def circular_distance(L, lag):
    d = np.abs(np.arange(L) - lag)
    return np.minimum(d, L - d)


def peak2_of(P, lag, excl):
    """The reduction of acq_peak2 over a power vector: (peak2, lag2 -- the lowest lag of the maximum --, ratio,
    noise_ex) over the lags at circular distance > excl from `lag`."""
    P = np.asarray(P)
    out = circular_distance(P.size, lag) > excl
    idx = np.nonzero(out)[0]
    i = idx[np.argmax(P[idx])]
    return P[i], int(i), P[lag] / P[i], P[idx].mean()
