"""Synthetic 1-bit (optionally 2-bit sign/magnitude) IF captures in the receiver's wire format (bench / smoke input data).

    s[i] = sum_k A_k * c_k(i + tau_k) * cos(2*pi*(FC + f_k)*i/FS + phi_k) + n[i],   n ~ N(0, 1)
    A_k  = sqrt(4 * 10^(CN0_k/10) / FS);   bit = (s < 0);   sample i -> bit (i & 7) of byte i >> 3

FS = 16.368 MHz, FC = 4.092 MHz (reference gps/gps.h:42-43), 65536 samples (8192 bytes) per block
(gps/gps.h:73, gps/search.cpp:389-411).  numpy on the host, or torch on a GPU for large batches.
This is host-side tooling: it does not touch the search path.
"""
import os

import numpy as np

from .sats import E1B

FS = 16.368e6
FC = 4.092e6
BLOCK_SAMPLES = 65536
BLOCK_BYTES = 8192

_DATA = os.path.join(os.path.dirname(os.path.abspath(__file__)), "data", "e1b_codes.bin")
_e1b_blob = None


def ca_chips(t1, t2):
    """1023 C/A chips (0/1).  G1 = 1+x^3+x^10, G2 = 1+x^2+x^3+x^6+x^8+x^9+x^10 (IS-GPS-200); rows with
    t1 or t2 > 10 give the G2 preset in t2 and tap stage 10 (QZSS/SBAS), as in the reference's table."""
    preset = t1 > 10 or t2 > 10
    g1 = [1] * 11
    g2 = [1] * 11
    if preset:
        for i in range(1, 11):
            g2[i] = (t2 >> (i - 1)) & 1
    out = np.zeros(1023, np.uint8)
    for n in range(1023):
        out[n] = (g1[10] ^ g2[10]) if preset else (g1[10] ^ g2[t1] ^ g2[t2])
        f1 = g1[3] ^ g1[10]
        f2 = g2[2] ^ g2[3] ^ g2[6] ^ g2[8] ^ g2[9] ^ g2[10]
        g1 = [0, f1] + g1[1:10]
        g2 = [0, f2] + g2[1:10]
    return out


def e1b_chips(prn):
    """4092 chips (0/1) of Galileo E1-B PRN prn (1..50) from the packed ICD table."""
    global _e1b_blob
    if _e1b_blob is None:
        _e1b_blob = np.fromfile(_DATA, np.uint8)
        assert _e1b_blob.size == 50 * 512
    rec = _e1b_blob[(prn - 1) * 512: prn * 512]
    return np.unpackbits(rec, bitorder="little")[:4092].copy()


def sat_chips(row):
    """(chips, boc) for a satellite-table row."""
    prn, t1, t2, typ = row
    if typ == E1B:
        return e1b_chips(prn), True
    return ca_chips(t1, t2), False


def _planes(s, sample_bits, mag_thr):
    """Quantise real samples s (noise sigma 1) to the capture wire format: sign bits, LSB first; with
    sample_bits == 2 every 65536-sample block is its sign plane followed by its magnitude plane
    (mag = |s| > mag_thr; include/acq_b200.h ACQ_CAPTURE_BLOCK_BYTES)."""
    sign = np.packbits(s < 0, bitorder="little")
    if sample_bits != 2:
        return sign
    mag = np.packbits(np.abs(s) > mag_thr, bitorder="little")
    return np.concatenate([sign.reshape(-1, 1, BLOCK_BYTES), mag.reshape(-1, 1, BLOCK_BYTES)], axis=1).reshape(-1)


F_L1 = 1575.42e6
BIT_SAMPLES = 327360   # one 20 ms GPS/QZSS L1 C/A data bit at FS


def make_capture(seed, n_blocks, sats, signals, sample_bits=1, mag_thr=0.98, code_doppler=False, chip_source=None,
                 data_bits=None, bit_edge=0):
    """numpy generator.  signals: iterable of (sat, tau, doppler_hz, cn0_dbhz, phase).  Returns uint8[n_blocks*8192]
    (sample_bits=2: uint8[n_blocks*16384], 2-bit sign/magnitude with the same sign bits; mag_thr in noise sigmas --
    0.98 is the optimum of a 4-level quantiser with levels +-1, +-3, a magnitude duty cycle of about 1/3).
    code_doppler=True also applies each signal's Doppler to its code rate (0.52 chip of drift over 80 ms at 10 kHz).
    chip_source: optional callable(row) -> (chips, boc) replacing this module's code tables (the golden generator passes
    the reference's own code classes, so that those fixtures do not depend on the product's tables).
    data_bits: optional GPS data-bit modulation of every non-E1B signal: a sequence of signs (+1 / -1), bit k covering
    samples [bit_edge + k BIT_SAMPLES, bit_edge + (k + 1) BIT_SAMPLES) (20 ms bits; k < 0 before bit_edge), taken
    cyclically.  None (the default) leaves the samples, and so the bytes, as without it."""
    rng = np.random.Generator(np.random.Philox(int(seed)))
    n = n_blocks * BLOCK_SAMPLES
    i = np.arange(n, dtype=np.int64)
    s = rng.standard_normal(n)
    for sat, tau, dop, cn0, phase in signals:
        chips, boc = (chip_source or sat_chips)(sats[sat])
        # code_doppler: the code is stretched by the carrier offset like a real signal's (f/f_L1 chips per chip)
        idx = (np.floor(i * (1.0 + dop / F_L1)).astype(np.int64) if code_doppler else i) + int(tau)
        c = chips[(idx >> 4) % len(chips)].astype(np.int8)
        if boc:
            c = c ^ ((idx & 15) >= 8)
        amp = np.sqrt(4.0 * 10.0 ** (cn0 / 10.0) / FS)
        cyc = (dop / FS * i) % 1.0 + 0.25 * (i & 3)
        if data_bits is not None and not boc:
            bits = np.asarray(data_bits, np.float64)
            amp = amp * bits[np.floor_divide(i - int(bit_edge), BIT_SAMPLES) % bits.size]
        s += amp * (1.0 - 2.0 * c) * np.cos(2.0 * np.pi * cyc + phase)
    return _planes(s, sample_bits, mag_thr)


def make_captures_torch(seed, n_captures, n_blocks, sats, signals_per_capture, device):
    """Batched torch generator (for the receiver-farm sizes).  signals_per_capture: list (len n_captures) of
    signal lists as in make_capture.  Returns a uint8 tensor [n_captures, n_blocks*8192] on `device`."""
    import torch

    g = torch.Generator(device=device)
    g.manual_seed(int(seed))
    n = n_blocks * BLOCK_SAMPLES
    i = torch.arange(n, device=device, dtype=torch.int64)
    out = torch.empty((n_captures, n // 8), dtype=torch.uint8, device=device)
    weights = (2 ** torch.arange(8, device=device, dtype=torch.int32)).to(torch.uint8)
    chip_cache = {}
    for c in range(n_captures):
        s = torch.randn(n, generator=g, device=device, dtype=torch.float64)
        for sat, tau, dop, cn0, phase in signals_per_capture[c]:
            if sat not in chip_cache:
                ch, boc = sat_chips(sats[sat])
                chip_cache[sat] = (torch.from_numpy(ch.astype(np.int64)).to(device), boc)
            ch, boc = chip_cache[sat]
            idx = i + int(tau)
            cc = ch[(idx >> 4) % ch.numel()]
            if boc:
                cc = cc ^ ((idx & 15) >= 8).to(torch.int64)
            amp = float(np.sqrt(4.0 * 10.0 ** (cn0 / 10.0) / FS))
            cyc = torch.remainder(dop / FS * i.to(torch.float64), 1.0) + 0.25 * (i & 3).to(torch.float64)
            s += amp * (1.0 - 2.0 * cc.to(torch.float64)) * torch.cos(2.0 * np.pi * cyc + phase)
        bits = (s < 0).to(torch.uint8).view(-1, 8)
        out[c] = (bits * weights).sum(dim=1, dtype=torch.int32).to(torch.uint8)
    return out


def make_capture_batch_torch(seeds, n_blocks, sats, signals_per_capture, device, group=64):
    """Batched torch generator with ONE SEED PER CAPTURE: capture i depends only on seeds[i] and its signal list, so a
    rank that generates just its shard of a sharded batch gets the same bytes as a rank that generates everything.
    Returns a uint8 tensor [len(seeds), n_blocks*8192] on `device`.  (Same signal model as make_capture; the noise
    comes from torch's generator, so the bytes differ from the numpy generator's for the same seed.)"""
    import torch

    n = n_blocks * BLOCK_SAMPLES
    n_cap = len(seeds)
    out = torch.empty((n_cap, n // 8), dtype=torch.uint8, device=device)
    i = torch.arange(n, device=device, dtype=torch.int64)
    fi = i.to(torch.float64)
    quarter = 0.25 * (i & 3).to(torch.float64)
    weights = (2 ** torch.arange(8, device=device, dtype=torch.int32)).to(torch.uint8)
    g = torch.Generator(device=device)
    chip_cache = {}
    for g0 in range(0, n_cap, group):
        g1 = min(n_cap, g0 + group)
        s = torch.empty((g1 - g0, n), dtype=torch.float64, device=device)
        for c in range(g0, g1):
            g.manual_seed(int(seeds[c]))
            s[c - g0] = torch.randn(n, generator=g, device=device, dtype=torch.float64)
            for sat, tau, dop, cn0, phase in signals_per_capture[c]:
                if sat not in chip_cache:
                    ch, boc = sat_chips(sats[sat])
                    chip_cache[sat] = (torch.from_numpy(1.0 - 2.0 * ch.astype(np.float64)).to(device), boc)
                ch, boc = chip_cache[sat]
                idx = i + int(tau)
                cc = ch[(idx >> 4) % ch.numel()]
                if boc:
                    cc = torch.where((idx & 15) >= 8, -cc, cc)
                amp = float(np.sqrt(4.0 * 10.0 ** (cn0 / 10.0) / FS))
                cyc = torch.remainder(dop / FS * fi, 1.0) + quarter
                s[c - g0] += amp * cc * torch.cos(2.0 * np.pi * cyc + phase)
        bits = (s < 0).to(torch.uint8).view(g1 - g0, -1, 8)
        out[g0:g1] = (bits * weights).sum(dim=2, dtype=torch.int32).to(torch.uint8)
    return out
