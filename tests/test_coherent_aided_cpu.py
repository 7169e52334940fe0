"""CPU suite for the aided coherent search (acq_search_coherent_aided / acq_search_coherent_aided_device): its argument
errors that need no engine are reported with a NULL engine, and CaptureFarm(m_coh=..., half_width=...) shards captures
and centres over the ranks -- no GPU needed."""
import ctypes as C
import os

import numpy as np

from flydog_sdr_gps_b200 import _lib

ENTRY_POINTS = ("acq_search_coherent_aided", "acq_search_coherent_aided_device")


def test_both_entry_points_are_exported_and_bound():
    L = _lib.load()
    names = _lib.exported_symbols()
    for n in ENTRY_POINTS:
        assert n in names and hasattr(L, n)


def _call(L, name, eng, m_coh, center, half_width):
    cap = np.zeros(8192, np.uint8)
    out = np.zeros(64, np.uint8)
    c = center.ctypes.data if center is not None else None
    # the last argument is the grid (host form) or the stream (device form): NULL for both
    return getattr(L, name)(eng, cap.ctypes.data, 1, None, 0, m_coh, c, half_width, out.ctypes.data, None)


def test_argument_errors_without_gpu():
    """A NULL dop_center, a negative half_width, m_coh outside 1..ACQ_COH_MAX and a window wider than any engine's
    coherent grid are ACQ_ERR_ARG (-1) with their own text, reported before the NULL engine is."""
    L = _lib.load()
    center = np.zeros(64, np.int32)
    for name in ENTRY_POINTS:
        assert _call(L, name, None, 2, center, 2) == -1
        assert b"engine is NULL" in L.acq_last_error()
        assert _call(L, name, None, 2, None, 2) == -1
        assert b"dop_center is NULL" in L.acq_last_error()
        assert _call(L, name, None, 2, center, -1) == -1
        assert b"half_width must be >= 0" in L.acq_last_error()
        for m in (0, 6, -1):
            assert _call(L, name, None, m, center, 2) == -1
            assert b"m_coh=%d outside 1..5" % m in L.acq_last_error()
        # n_dop_c <= 5 * 8188 + 1 for every engine; also keeps 2 * half_width + 1 from overflowing
        for hw in (5 * 4094 + 1, 2 ** 31 - 1):
            assert _call(L, name, None, 5, center, hw) == -1
            assert b"exceeds n_dop_c" in L.acq_last_error()


class _TagEngine:
    """Stand-in for AcqEngine in CaptureFarm: search_coherent_aided_device writes, for each row, the capture's tag (its
    first byte) into lag, the row's centre into dop and m_coh * 1000 + half_width into sat.  The gathered records then
    show which rank searched which captures with which centres."""
    device = "cpu"

    def __init__(self, n_sel, capture_bytes):
        self.n_sel, self.capture_bytes = n_sel, capture_bytes

    def search_coherent_aided_device(self, packed_dev, m_coh, dop_center_dev, half_width, out_dev, n_cap, sel=None,
                                     stream_ptr=None):
        from flydog_sdr_gps_b200.engine import RECORD_DTYPE
        packed = np.ctypeslib.as_array((C.c_uint8 * (n_cap * self.capture_bytes)).from_address(packed_dev))
        centers = np.ctypeslib.as_array((C.c_int32 * (n_cap * self.n_sel)).from_address(dop_center_dev))
        out = np.ctypeslib.as_array((C.c_uint8 * (n_cap * self.n_sel * 24)).from_address(out_dev)).view(RECORD_DTYPE)
        for c in range(n_cap):
            for s in range(self.n_sel):
                r = out[c * self.n_sel + s]
                r["sat"], r["lag"], r["dop"] = m_coh * 1000 + half_width, packed[c * self.capture_bytes], centers[c * self.n_sel + s]


def _worker(rank, world, port, caps, centers, out_dir):
    import torch.distributed as dist
    from flydog_sdr_gps_b200 import farm
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    n_cap, n_sel = centers.shape
    f = farm.CaptureFarm(_TagEngine(n_sel, caps.shape[1]), n_cap, caps.shape[1], n_sel, dist=dist, device="cpu",
                         m_coh=4, half_width=7)
    f.load(caps, dop_center=centers)
    rec = f.search().copy()
    assert np.array_equal(f.search_resident().numpy(), f.h_all.numpy())
    np.save(os.path.join(out_dir, "rank_%d.npy" % rank), rec)
    dist.barrier()
    dist.destroy_process_group()


def test_capture_farm_coherent_aided_world_size_2(tmp_path):
    """3 captures over 2 ranks (uneven shards, padded gather): every rank returns [3, n_sel] records in which row (c, s)
    carries capture c's tag and its own centre."""
    import socket
    import torch.multiprocessing as mp
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    n_cap, n_sel, nbytes = 3, 5, 2 * 8192
    caps = np.zeros((n_cap, nbytes), np.uint8)
    caps[:, 0] = [11, 22, 33]
    centers = (np.arange(n_cap * n_sel, dtype=np.int32).reshape(n_cap, n_sel) * 7 - 40)
    mp.spawn(_worker, args=(2, port, caps, centers, str(tmp_path)), nprocs=2, join=True)
    for r in range(2):
        got = np.load(os.path.join(str(tmp_path), "rank_%d.npy" % r))
        assert got.shape == (n_cap, n_sel)
        assert np.array_equal(got["lag"], np.repeat([[11], [22], [33]], n_sel, axis=1))
        assert np.array_equal(got["dop"], centers)
        assert np.all(got["sat"] == 4 * 1000 + 7)
