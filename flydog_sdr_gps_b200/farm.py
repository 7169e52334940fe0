"""Multi-GPU plumbing: one process per GPU, independent units sharded across ranks, only the small
record arrays gathered (SURVEY.md 8(e)).  No data-path collective exists on this path: the (capture, sat,
Doppler) tiles share nothing but read-only inputs, and the only cross-tile step -- best-over-Doppler per
(capture, sat) -- stays on the GPU that owns the pair.

  CaptureFarm (receiver farm, cfg5)  : every rank holds all code spectra and searches its slice of the captures
  SatFarm     (one capture, cfg4)    : the capture is given to every rank, each searches a slice of the table

Both keep their buffers for the life of the object (pinned host staging, device captures, device records, the gathered
record array), so a search is: host->device copy of the local captures, acq_search_device on the current torch stream,
all_gather_into_tensor of the 24-byte records over NCCL, device->host copy of the gathered array.  `search_resident`
is the same without the two copies (captures already in HBM, records left there).

`engine` is an AcqEngine.  The CPU suite exercises the same classes under gloo with a stand-in whose
`search_device(...)` runs the oracle on CPU tensors; nothing in this module computes a search itself.
The function forms below (`search_sharded_by_*`) are the numpy/host-gather variant of the same plumbing.
"""
import numpy as np

from .engine import RECORD_DTYPE
from .scenarios import shard

REC = RECORD_DTYPE.itemsize


class _Farm:
    def __init__(self, engine, n_units, dist=None, device=None):
        import torch
        self.torch = torch
        self.eng = engine
        self.dist = dist
        self.rank, self.world = (dist.get_rank(), dist.get_world_size()) if dist is not None else (0, 1)
        self.device = torch.device(device) if device is not None else torch.device("cuda", engine.device)
        self.n_units = n_units
        self.lo, self.hi = shard(n_units, self.rank, self.world)
        self.n_local = self.hi - self.lo
        self.counts = [shard(n_units, r, self.world)[1] - shard(n_units, r, self.world)[0] for r in range(self.world)]
        self.max_local = max(self.counts)
        self.pin = self.device.type == "cuda"

    def _empty(self, n, device=None, pin=False):
        t = self.torch.zeros(max(n, 1), dtype=self.torch.uint8, device=device or self.device)
        return t.pin_memory() if pin else t

    def _stream_ptr(self):
        return self.torch.cuda.current_stream().cuda_stream if self.device.type == "cuda" else None

    def _gather(self):
        """Padded all_gather of the local record bytes; afterwards self.d_all holds every rank's slot."""
        if self.world > 1:
            self.dist.all_gather_into_tensor(self.d_all, self.d_rec)

    def _unpad(self, host_bytes, per_unit):
        """host_bytes: uint8 numpy [world * max_local * per_unit * REC] -> records in unit order."""
        slot = self.max_local * per_unit * REC
        parts = [host_bytes[r * slot: r * slot + self.counts[r] * per_unit * REC] for r in range(self.world)]
        return np.concatenate(parts).view(RECORD_DTYPE)


class CaptureFarm(_Farm):
    """n_captures independent captures (each `capture_bytes` long) sharded over the ranks; the whole table is searched on
    each.  Records come back as [n_captures, n_sel] on every rank.

    half_width (optional): an aided farm -- every (capture, satellite) row searches only the 2 * half_width + 1 Doppler
    indices around its own centre (acq_search_aided_device); load() then takes the centres with the captures."""

    def __init__(self, engine, n_captures, capture_bytes, n_sel, dist=None, device=None, half_width=None):
        super().__init__(engine, n_captures, dist, device)
        self.capture_bytes, self.n_sel = capture_bytes, n_sel
        self.half_width = half_width
        self.h_in = self._empty(self.n_local * capture_bytes, device="cpu", pin=self.pin)
        self.d_in = self._empty(self.n_local * capture_bytes)
        if half_width is not None:   # this rank's Doppler centres, int32 [n_local, n_sel], kept in HBM with the captures
            self.d_center = self.torch.zeros(max(self.n_local * n_sel, 1), dtype=self.torch.int32, device=self.device)
        self.d_rec = self._empty(self.max_local * n_sel * REC)           # local records, padded to the largest shard
        self.d_all = self._empty(self.world * self.max_local * n_sel * REC) if self.world > 1 else self.d_rec
        self.h_all = self._empty(self.d_all.numel(), device="cpu", pin=self.pin)

    def load(self, captures, dop_center=None):
        """captures: uint8 numpy [n_captures, capture_bytes] (every rank may pass the whole set) or just this rank's
        [n_local, capture_bytes] slice.  Stages the local slice in pinned memory and in HBM.  dop_center (aided farm
        only, required there): int [n_captures, n_sel] or this rank's [n_local, n_sel], sharded like the captures."""
        a = np.ascontiguousarray(captures, np.uint8).reshape(-1, self.capture_bytes)
        if a.shape[0] == self.n_units:
            a = a[self.lo:self.hi]
        assert a.shape[0] == self.n_local, (a.shape, self.n_local)
        if (dop_center is None) != (self.half_width is None):
            raise ValueError("dop_center is given exactly when the farm was created with half_width")
        if dop_center is not None:
            c = np.ascontiguousarray(dop_center, np.int32).reshape(-1, self.n_sel)
            if c.shape[0] == self.n_units:
                c = c[self.lo:self.hi]
            assert c.shape[0] == self.n_local, (c.shape, self.n_local)
            if self.n_local:
                self.d_center[:c.size].copy_(self.torch.from_numpy(c.reshape(-1)))
        if self.n_local:
            self.h_in[:a.size].copy_(self.torch.from_numpy(a.reshape(-1)))
            self.d_in.copy_(self.h_in)

    def search_resident(self):
        """Captures (and, aided, centres) already in HBM (load()); leaves the gathered records in self.d_all.  Asynchronous."""
        if self.n_local and self.half_width is not None:
            self.eng.search_aided_device(self.d_in.data_ptr(), self.d_center.data_ptr(), self.half_width, self.d_rec.data_ptr(),
                                         self.n_local, stream_ptr=self._stream_ptr())
        elif self.n_local:
            self.eng.search_device(self.d_in.data_ptr(), self.d_rec.data_ptr(), self.n_local, stream_ptr=self._stream_ptr())
        self._gather()
        return self.d_all

    def search(self):
        """End to end from the pinned host captures: copy in, search, gather, copy out, wait.  Returns records
        [n_captures, n_sel] (numpy view of the pinned result buffer: valid until the next search)."""
        if self.n_local:
            self.d_in.copy_(self.h_in, non_blocking=True)
        self.search_resident()
        self.h_all.copy_(self.d_all, non_blocking=True)
        if self.device.type == "cuda":
            self.torch.cuda.current_stream().synchronize()
        return self._unpad(self.h_all.numpy(), self.n_sel).reshape(self.n_units, self.n_sel)

    @property
    def h2d_bytes(self):
        return self.n_local * self.capture_bytes

    @property
    def d2h_bytes(self):
        return int(self.d_all.numel())


class SatFarm(_Farm):
    """ONE capture, the satellite table sharded over the ranks (the loop `for (sp = Sats; ...)` of gps/search.cpp:530 is
    what is being split: each satellite's whole Doppler scan, with its first-wins tie-break, stays on one GPU).
    Records come back as [n_sats] in table order on every rank."""

    def __init__(self, engine, n_sats, capture_bytes, dist=None, device=None):
        super().__init__(engine, n_sats, dist, device)
        self.capture_bytes = capture_bytes
        self.sel = np.arange(self.lo, self.hi, dtype=np.int32)
        self.h_in = self._empty(capture_bytes, device="cpu", pin=self.pin)
        self.d_in = self._empty(capture_bytes)
        self.d_rec = self._empty(self.max_local * REC)
        self.d_all = self._empty(self.world * self.max_local * REC) if self.world > 1 else self.d_rec
        self.h_all = self._empty(self.d_all.numel(), device="cpu", pin=self.pin)

    def load(self, capture):
        a = np.ascontiguousarray(capture, np.uint8).reshape(-1)
        assert a.size == self.capture_bytes
        self.h_in.copy_(self.torch.from_numpy(a))
        self.d_in.copy_(self.h_in)

    def search_resident(self):
        if self.n_local:
            self.eng.search_device(self.d_in.data_ptr(), self.d_rec.data_ptr(), 1, sel=self.sel, stream_ptr=self._stream_ptr())
        self._gather()
        return self.d_all

    def search(self):
        self.d_in.copy_(self.h_in, non_blocking=True)   # the capture is broadcast by giving it to every rank
        self.search_resident()
        self.h_all.copy_(self.d_all, non_blocking=True)
        if self.device.type == "cuda":
            self.torch.cuda.current_stream().synchronize()
        return self._unpad(self.h_all.numpy(), 1)

    @property
    def h2d_bytes(self):
        return self.capture_bytes

    @property
    def d2h_bytes(self):
        return int(self.d_all.numel())


# ---- host-gather function forms (numpy records, all_gather of padded byte tensors) -------------------------------
def _gather_records(local, counts, dist, device):
    """all_gather of variable-length record arrays as padded uint8 tensors; returns list per rank."""
    import torch
    world = dist.get_world_size()
    width = max(counts) * REC
    buf = np.zeros(width, np.uint8)
    raw = local.reshape(-1).view(np.uint8)
    buf[:raw.size] = raw
    t = torch.from_numpy(buf).to(device)
    out = [torch.empty_like(t) for _ in range(world)]
    dist.all_gather(out, t)
    return [o.cpu().numpy()[:counts[r] * REC].view(RECORD_DTYPE) for r, o in enumerate(out)]


def search_sharded_by_capture(search_fn, captures, n_sel, dist=None, device="cpu"):
    """captures: uint8 [n_cap, bytes].  search_fn(captures_slice) -> records [n, n_sel].  Returns records
    [n_cap, n_sel] (on every rank)."""
    n_cap = captures.shape[0]
    rank, world = (dist.get_rank(), dist.get_world_size()) if dist is not None else (0, 1)
    lo, hi = shard(n_cap, rank, world)
    local = search_fn(captures[lo:hi]) if hi > lo else np.zeros((0, n_sel), RECORD_DTYPE)
    if world == 1:
        return local
    counts = [(shard(n_cap, r, world)[1] - shard(n_cap, r, world)[0]) * n_sel for r in range(world)]
    parts = _gather_records(local, counts, dist, device)
    return np.concatenate([p.reshape(-1, n_sel) for p in parts], axis=0)


def search_sharded_by_sat(search_fn, capture, n_sats, dist=None, device="cpu"):
    """One capture, satellite table split across ranks.  search_fn(capture, sel) -> records [len(sel)].
    Returns records [n_sats] in table order (on every rank)."""
    rank, world = (dist.get_rank(), dist.get_world_size()) if dist is not None else (0, 1)
    lo, hi = shard(n_sats, rank, world)
    local = search_fn(capture, np.arange(lo, hi, dtype=np.int32)) if hi > lo else np.zeros(0, RECORD_DTYPE)
    if world == 1:
        return local
    counts = [shard(n_sats, r, world)[1] - shard(n_sats, r, world)[0] for r in range(world)]
    return np.concatenate(_gather_records(local, counts, dist, device))
