"""Reference side of the peak-quality tests (acq_profile): the power vector that the oracle's Correlate restatement
(oracle/acq_oracle.c, correlate_one) forms at one Doppler index, summed over the K blocks, rebuilt from the oracle's own
exported stages -- capture baseband, code spectrum, 16384-point FFT -- with nothing new but the indexing; and the
second-peak reduction over such a vector."""
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


def orc_profile(O, params, capture, sats, sat, dop):
    """float64 [L]: sum over the K blocks of |r_b[(n + 16 b + s(b, dop)) mod N]|^2 (s = 0 without code_doppler; for K = 1
    just |r[n]|^2), r_b = IFFT(conj(D_b) * code[(k - d) mod N]) with correlate_one's row addressing: for a negative
    Doppler the bins past the end of the doubled row come from the next table row (reference wrap, zeros after the last
    row) or from the same row (circular wrap).  dop is the Doppler index (half-bins when half_bin)."""
    K, half_bin = int(params.k_noncoh), int(params.half_bin)
    bits = int(params.sample_bits) or 1
    bb = O.block_bytes(bits)
    v = (dop & 1) if half_bin else 0
    d = (dop - v) // 2 if half_bin else dop
    C = O.code_spectrum(sats[sat])
    nxt = O.code_spectrum(sats[sat + 1]) if sat + 1 < len(sats) else np.zeros(N, np.complex64)
    j = np.arange(N) - d
    code = C[j % N].copy()
    past = j >= N   # only for d < 0
    if params.wrap_mode == O.WRAP_REFERENCE:
        code[past] = nxt[j[past] - N]
    L = LAGS_E1B if sats[sat][3] == E1B else LAGS_L1
    cap = np.ascontiguousarray(capture, np.uint8).reshape(-1)
    P = np.zeros(L, np.float64)
    n = np.arange(L)
    for b in range(K):
        D = O.fft16384(O.capture_baseband(cap[b * bb:(b + 1) * bb], half_rot=v, sample_bits=bits), -1)
        r = O.fft16384(np.conj(D) * code, +1).astype(np.complex128)
        cs = code_shift(b, dop, half_bin) if params.code_doppler else 0
        m = (n + (16 * b + cs if K > 1 else 0)) % N
        P += np.abs(r[m]) ** 2
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
