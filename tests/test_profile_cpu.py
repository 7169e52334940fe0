"""CPU suite for the peak-quality profile (acq_profile / acq_profile_device): exports and struct layout, the argument
errors that need no engine state, the oracle-side reference against the oracle's own search, and the farms' profile()
under gloo with world size 2 -- no GPU needed."""
import ctypes as C
import os
import socket
import subprocess

import numpy as np
import pytest

from flydog_sdr_gps_b200 import _lib, engine, synth
from flydog_sdr_gps_b200 import sats as S

from profile_ref import LAGS_L1, orc_profile, peak2_of

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_entry_points_are_exported_and_bound():
    L = _lib.load()
    for name in ("acq_profile", "acq_profile_device"):
        assert name in _lib.exported_symbols() and hasattr(L, name)
    assert hasattr(engine.AcqEngine, "profile") and hasattr(engine.AcqEngine, "profile_device")
    assert engine.PROFILE_DETECTED == 1
    assert engine.PEAK2_DTYPE.itemsize == 16 and engine.PEAK2_DTYPE.names == ("peak2", "lag2", "ratio", "noise_ex")


def test_peak2_layout_matches_header(tmp_path):
    """sizeof / offsets of acq_peak2 as a C compiler sees include/acq_b200.h, against PEAK2_DTYPE."""
    src = tmp_path / "layout.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "acq_b200.h"\n'
                   'int main(void) { printf("%zu %zu %zu %zu %zu %d\\n", sizeof(acq_peak2), offsetof(acq_peak2, peak2), '
                   'offsetof(acq_peak2, lag2), offsetof(acq_peak2, ratio), offsetof(acq_peak2, noise_ex), '
                   'ACQ_PROFILE_DETECTED); return 0; }\n')
    exe = tmp_path / "layout"
    subprocess.run(["cc", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)], check=True)
    got = [int(v) for v in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    dt = engine.PEAK2_DTYPE
    assert got == [dt.itemsize] + [dt.fields[n][1] for n in dt.names] + [engine.PROFILE_DETECTED]


def test_argument_errors_without_gpu():
    """A NULL engine, NULL rec/out, a negative excl and unknown flag bits are ACQ_ERR_ARG (-1), each with its own text,
    before the engine is read."""
    L = _lib.load()
    rec = np.zeros(64, np.uint8)
    out = np.zeros(64, np.uint8)
    r, o = rec.ctypes.data, out.ctypes.data
    assert L.acq_profile(None, r, 2, 4, o, None) == -1
    assert b"engine is NULL" in L.acq_last_error()
    assert L.acq_profile_device(None, r, 2, 0, 4, o, None, None) == -1
    assert b"engine is NULL" in L.acq_last_error()
    fake = C.c_void_p(o)   # any non-NULL handle: these checks come before the engine is read
    assert L.acq_profile(fake, None, 2, 4, o, None) == -1
    assert b"rec/out must not be NULL" in L.acq_last_error()
    assert L.acq_profile(fake, r, 2, 4, None, None) == -1
    assert b"rec/out must not be NULL" in L.acq_last_error()
    assert L.acq_profile(fake, r, 2, -1, o, None) == -1
    assert b"excl must be >= 0" in L.acq_last_error()
    assert L.acq_profile_device(fake, None, 2, 0, 4, o, None, None) == -1
    assert b"rec_dev/out_dev must not be NULL" in L.acq_last_error()
    assert L.acq_profile_device(fake, r, 2, 0, 4, None, None, None) == -1
    assert b"rec_dev/out_dev must not be NULL" in L.acq_last_error()
    for flags in (2, 0x100, -1):
        assert L.acq_profile_device(fake, r, 2, flags, 4, o, None, None) == -1
        assert b"unknown flag bits" in L.acq_last_error()
    assert L.acq_profile_device(fake, r, 2, 0, -3, o, None, None) == -1
    assert b"excl must be >= 0" in L.acq_last_error()


_GRID_CASES = {
    # (table, oracle params, blocks, signals, sel, sample_bits, code-Doppler capture)
    "reference_wrap": ("nav", {}, 1, [(3, 2000, 5.4 * engine.BIN_HZ, 47, 0.3), (31, 9000, -11.2 * engine.BIN_HZ, 47, 1.0)],
                       [3, 30, 31], 1, False),
    "circular_wrap": ("nav", dict(wrap_mode=1), 1, [(30, 700, -8.0 * engine.BIN_HZ, 47, 0.3)], [30, 31], 1, False),
    "half_bin_k3_code_doppler": ("nav", dict(k_noncoh=3, half_bin=1, dop_lo=-25, dop_hi=24, code_doppler=1), 3,
                                 [(3, 2000, 5.4 * engine.BIN_HZ, 47, 0.3), (8, 640, -4.3 * engine.BIN_HZ, 45, 2.0)],
                                 [3, 8], 1, True),
    "sample_bits_2": ("nav", dict(sample_bits=2), 1, [(12, 333, -3.0 * engine.BIN_HZ, 46, 0.7)], [12, 13], 2, False),
    "e1b_k2": ("e1b", dict(k_noncoh=2, dop_lo=-6, dop_hi=5), 2, [(1, 30001, -3.0 * engine.BIN_HZ, 48, 0.1)], [1, 4], 1,
               False),
}


@pytest.mark.parametrize("case", sorted(_GRID_CASES))
def test_reference_profile_agrees_with_the_oracle_grid(oracle, case):
    """orc_profile against the oracle's own search at EVERY Doppler cell of its grid (negative Dopplers with the next
    table row or the circular wrap, the last table row's zero neighbour, odd half-bin indices, code-Doppler shifts of a
    K-block sum, 2-bit captures, E1B): the vector's first maximum is the cell's lag, its maximum the cell's peak and its
    mean the cell's noise -- a check of the restatement's row addressing, not only at the detected Doppler."""
    which, kw, blocks, sig, sel, bits, cd = _GRID_CASES[case]
    table = S.navstar() if which == "nav" else S.e1b(range(1, 6))
    p = oracle.default_params(**kw)
    cap = synth.make_capture(17, blocks, table, sig, sample_bits=bits, code_doppler=cd)
    rec, grid = oracle.search(cap, table, sel=sel, params=p, want_grid=True, nthreads=1)
    for s, sat in enumerate(sel):
        for d in range(grid.shape[1]):
            cell = grid[s, d]
            P = orc_profile(oracle, p, cap, table, sat, p.dop_lo + d)
            assert P.size == (LAGS_L1 if which == "nav" else 16368)
            m = P.max()
            assert abs(m - cell["peak"]) <= 1e-5 * cell["peak"], (case, sat, d)
            assert int(np.argmax(P)) == cell["lag"] or P[cell["lag"]] >= m * (1 - 1e-5), (case, sat, d)
            assert abs(P.mean() - cell["noise"]) <= 2e-4 * cell["noise"], (case, sat, d)
        assert rec[s]["peak"] == grid[s, rec[s]["dop"] - p.dop_lo]["peak"]


def test_peak2_reduction():
    P = np.ones(100)
    P[10], P[12], P[60], P[95] = 50.0, 30.0, 7.0, 7.0
    assert peak2_of(P, 10, 2) == (7.0, 60, 50.0 / 7.0, (P.sum() - 50 - 30 - 3) / 95)   # lobe 8..12
    P[8] = 9.0   # inside the lobe of 10 at excl 2; at excl 1 the shoulder at 12 is outside it and is the second peak
    assert peak2_of(P, 10, 2)[1] == 60 and peak2_of(P, 10, 1)[:2] == (30.0, 12)
    assert peak2_of(P, 95, 5)[1] == 10   # circular: lags 0..2 and 90..99 are the lobe of 95
    assert peak2_of(P, 1, 3)[1] == 10   # the main peak of another lag is just the largest power outside the lobe


# ---- farms under gloo: sharding / padding / gather of the 16-byte rows, the oracle as the engine
THR = 16.0
EXCL = 4
NAN = np.array([0x7fc00000], np.uint32).view(np.float32)[0]   # the quiet NaN the kernel writes into marker rows


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def oracle_peak2(O, caps, table, rec, excl, detected_only):
    """PEAK2_DTYPE rows of records [n_cap, n_sel] from the oracle's profiles; undetected rows get the -1 marker."""
    p = O.default_params()
    out = np.zeros(rec.shape, engine.PEAK2_DTYPE)
    for c in range(rec.shape[0]):
        for s in range(rec.shape[1]):
            r = rec[c, s]
            if detected_only and not r["snr"] >= THR:
                out[c, s] = (NAN, -1, NAN, NAN)
                continue
            P = orc_profile(O, p, caps[c], table, int(r["sat"]), int(r["dop"]))
            out[c, s] = peak2_of(P, int(r["lag"]), excl)
    return out


class _OracleEngine:
    """Stand-in for AcqEngine in the farm classes: search_device and profile_device with AcqEngine's signatures, the
    oracle as searcher and profile, CPU tensors as the 'device'.  profile_device evaluates the rows of its last search."""

    def __init__(self, table):
        from oracle import oracle_py as O
        self.O, self.table, self.device = O, table, "cpu"
        self.last = None

    def search_device(self, packed_ptr, out_ptr, n_cap, sel=None, stream_ptr=None):
        n_sel = len(self.table) if sel is None else len(sel)
        packed = np.ctypeslib.as_array((C.c_uint8 * (n_cap * 8192)).from_address(packed_ptr)).reshape(n_cap, 8192).copy()
        out = np.ctypeslib.as_array((C.c_uint8 * (n_cap * n_sel * 24)).from_address(out_ptr))
        rec = np.stack([self.O.search(c, self.table, sel=sel, nthreads=1) for c in packed])
        out[:] = rec.reshape(-1).view(np.uint8)
        self.last = (packed, n_sel)

    def profile_device(self, rec_dev, out_dev, n, excl=4, detected_only=False, profile_dev=None, stream_ptr=None):
        if self.last is None or n != len(self.last[0]) * self.last[1]:
            raise engine.AcqError(-1, "no search whose spectra are still on the device / wrong count")
        packed, n_sel = self.last
        rec = np.ctypeslib.as_array((C.c_uint8 * (n * 24)).from_address(rec_dev)).copy().view(engine.RECORD_DTYPE)
        pk = oracle_peak2(self.O, packed, self.table, rec.reshape(len(packed), n_sel), excl, detected_only)
        out = np.ctypeslib.as_array((C.c_uint8 * (n * 16)).from_address(out_dev))
        out[:] = pk.reshape(-1).view(np.uint8)


def _worker(rank, world, port, mode, caps, out_dir):
    import torch.distributed as dist
    from flydog_sdr_gps_b200 import farm
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    table = S.navstar()[:6]
    if mode == "capture_farm":   # 3 captures over 2 ranks: uneven shards, padded gather
        f = farm.CaptureFarm(_OracleEngine(table), len(caps), 8192, len(table), dist=dist, device="cpu")
        f.load(caps)
    else:                        # 5 satellites over 2 ranks
        f = farm.SatFarm(_OracleEngine(table[:5]), 5, 8192, dist=dist, device="cpu")
        f.load(caps[0])
    with pytest.raises(engine.AcqError):   # nothing searched on this farm yet
        f.profile()
    rec = f.search().copy()
    pk_all = f.profile(excl=EXCL, detected_only=False).copy()
    pk_det = f.profile(excl=EXCL).copy()
    assert np.array_equal(f.profile_resident(excl=EXCL).numpy(), f.h_pk_all.numpy())
    for name, a in (("rec", rec), ("all", pk_all), ("det", pk_det)):
        np.save(os.path.join(out_dir, "%s_%s_%d.npy" % (mode, name, rank)), a)
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("mode", ["capture_farm", "sat_farm"])
def test_world_size_2_profile_equals_single_process(tmp_path, mode, oracle):
    import torch.multiprocessing as mp
    table = S.navstar()[:6]
    caps = np.stack([synth.make_capture(s, 1, table, [(s % 6, 400 * s, 250.0 * s, 48, 0.1)]) for s in range(1, 4)])
    port = _free_port()
    mp.spawn(_worker, args=(2, port, mode, caps, str(tmp_path)), nprocs=2, join=True)
    if mode == "capture_farm":
        rec = np.stack([oracle.search(c, table, nthreads=1) for c in caps])
        want_all = oracle_peak2(oracle, caps, table, rec, EXCL, False)
        want_det = oracle_peak2(oracle, caps, table, rec, EXCL, True)
    else:
        rec = oracle.search(caps[0], table[:5], nthreads=1)
        want_all = oracle_peak2(oracle, caps[:1], table[:5], rec[None], EXCL, False)[0]
        want_det = oracle_peak2(oracle, caps[:1], table[:5], rec[None], EXCL, True)[0]
    want = {"rec": rec, "all": want_all, "det": want_det}
    assert (want_det["lag2"] == -1).any() and (want_det["lag2"] >= 0).any()
    assert np.isfinite(want_all["ratio"]).all() and (want_all["lag2"] >= 0).all()
    for r in range(2):
        for name, w in want.items():
            got = np.load(os.path.join(str(tmp_path), "%s_%s_%d.npy" % (mode, name, r)))
            assert got.shape == w.shape, (name, got.shape, w.shape)
            assert got.tobytes() == w.tobytes(), name
