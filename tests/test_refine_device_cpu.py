"""CPU suite for the device-resident refinement (acq_refine_device): exported by the library and the binding, its
argument errors that need no engine state, and the farms' refine() under gloo with world size 2 -- no GPU needed."""
import ctypes as C
import os
import socket

import numpy as np
import pytest

from flydog_sdr_gps_b200 import _lib, engine, synth
from flydog_sdr_gps_b200 import sats as S


def test_entry_point_is_exported_and_bound():
    L = _lib.load()
    assert "acq_refine_device" in _lib.exported_symbols() and hasattr(L, "acq_refine_device")
    assert hasattr(engine.AcqEngine, "refine_device") and engine.REFINE_DETECTED == 1


def test_argument_errors_without_gpu():
    """A NULL engine, a NULL rec_dev or out_dev and unknown flag bits are ACQ_ERR_ARG (-1), each with its own text."""
    L = _lib.load()
    rec = np.zeros(64, np.uint8)
    out = np.zeros(64, np.uint8)
    r, o = rec.ctypes.data, out.ctypes.data
    assert L.acq_refine_device(None, r, 2, 0, o, None) == -1
    assert b"engine is NULL" in L.acq_last_error()
    # any non-NULL handle: the pointer and flag checks come before the engine is read
    fake = C.c_void_p(o)
    assert L.acq_refine_device(fake, None, 2, 0, o, None) == -1
    assert b"rec_dev/out_dev must not be NULL" in L.acq_last_error()
    assert L.acq_refine_device(fake, r, 2, 0, None, None) == -1
    assert b"rec_dev/out_dev must not be NULL" in L.acq_last_error()
    for flags in (2, 0x100, -1):
        assert L.acq_refine_device(fake, r, 2, flags, o, None) == -1
        assert b"unknown flag bits" in L.acq_last_error()


# ---- farms under gloo: the sharding / padding / gather of the fine records, the oracle as the engine
THR = 16.0
NAN = np.array([0x7fc00000], np.uint32).view(np.float32)[0]   # the quiet NaN the kernel writes into marker rows


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _mark_undetected(fine, rec):
    """The ACQ_REFINE_DETECTED marker on every row below the threshold (the table here is all C/A)."""
    low = ~(rec["snr"] >= THR)
    fine["dop_hz"][low] = NAN
    fine["code_fs"][low] = NAN
    fine["peak"][low] = 0.0
    fine["ca_shift"][low] = -1
    return fine


class _OracleEngine:
    """Stand-in for AcqEngine in the farm classes: search_device and refine_device with AcqEngine's signatures, the
    oracle as searcher and refiner, CPU tensors as the 'device'.  refine_device refines the rows of its last search,
    which it remembers the way the engine keeps that search's spectra."""

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

    def refine_device(self, rec_dev, out_dev, n_records, detected_only=False, stream_ptr=None):
        if self.last is None or n_records != len(self.last[0]) * self.last[1]:
            raise engine.AcqError(-1, "no search whose spectra are still on the device / wrong count")
        packed, n_sel = self.last
        rec = np.ctypeslib.as_array((C.c_uint8 * (n_records * 24)).from_address(rec_dev)).copy().view(engine.RECORD_DTYPE)
        rec = rec.reshape(len(packed), n_sel)
        fine = np.stack([self.O.refine(c, self.table, r, nthreads=1) for c, r in zip(packed, rec)])
        if detected_only:
            fine = _mark_undetected(fine, rec)
        out = np.ctypeslib.as_array((C.c_uint8 * (n_records * 16)).from_address(out_dev))
        out[:] = fine.reshape(-1).view(np.uint8)


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
        f.refine()
    rec = f.search().copy()
    fine_all = f.refine(detected_only=False).copy()
    fine_det = f.refine().copy()
    assert np.array_equal(f.refine_resident().numpy(), f.h_fine_all.numpy())
    for name, a in (("rec", rec), ("all", fine_all), ("det", fine_det)):
        np.save(os.path.join(out_dir, "%s_%s_%d.npy" % (mode, name, rank)), a)
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("mode", ["capture_farm", "sat_farm"])
def test_world_size_2_refine_equals_single_process(tmp_path, mode, oracle):
    import torch.multiprocessing as mp
    table = S.navstar()[:6]
    caps = np.stack([synth.make_capture(s, 1, table, [(s % 6, 400 * s, 250.0 * s, 48, 0.1)]) for s in range(1, 4)])
    port = _free_port()
    mp.spawn(_worker, args=(2, port, mode, caps, str(tmp_path)), nprocs=2, join=True)
    if mode == "capture_farm":
        rec = np.stack([oracle.search(c, table, nthreads=1) for c in caps])
        fine = np.stack([oracle.refine(c, table, r, nthreads=1) for c, r in zip(caps, rec)])
    else:
        rec = oracle.search(caps[0], table[:5], nthreads=1)
        fine = oracle.refine(caps[0], table[:5], rec, nthreads=1)
    want = {"rec": rec, "all": fine, "det": _mark_undetected(fine.copy(), rec)}
    assert (want["det"]["ca_shift"] == -1).any() and (want["det"]["ca_shift"] >= 0).any()
    for r in range(2):
        for name, w in want.items():
            got = np.load(os.path.join(str(tmp_path), "%s_%s_%d.npy" % (mode, name, r)))
            assert got.shape == w.shape, (name, got.shape, w.shape)
            assert got.tobytes() == w.tobytes(), name
