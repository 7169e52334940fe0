#!/usr/bin/env python3
"""bench.py -- acquisition cells/s of the B200 engine on BASELINE.json's workloads.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

A "step" is one pass of the hot path (front end + PRN x Doppler x code-phase search + best-Doppler pick) over one
batch of synthetic captures.

HEADLINE line = BASELINE configs[4], the receiver farm (cfg5): 1024 independent captures x 32 GPS PRNs x 41 Doppler bins
(the reference's own search parameters, gps/search.cpp:465,530), 1024 captures IN TOTAL at every N -- strong scaling:
rank r searches scenarios.shard(1024, r, N) through farm.CaptureFarm (the CUDA engine behind the C ABI) and the 24-byte
records are gathered with NCCL inside the timed region.
  value      whole-job cells/s with the captures already resident in HBM (CUDA events, max over ranks)
  e2e        the same through host buffers: pinned captures -> H2D -> search -> NCCL gather -> D2H of all records
  configs    cfg1..cfg4 of BASELINE.json, each from its own CUDA-event loop.  N = 1: one GPU, `e2e` through acq_search()
             (the reference-facing C-ABI call, host buffers).  N > 1: the satellite list of the ONE capture is sharded
             over the ranks (farm.SatFarm: capture given to every rank, records gathered) -- cfg4_prn_sharded is
             BASELINE configs[3]; these are latency-bound by launch + gather, as SURVEY 8(e) predicts.
  roofline   dominant kernel (fused correlate + inverse FFT + peak search) against the on-SM roofs measured by
             micro-benchmark in this run and against measured HBM; `frac` = the shared-memory bytes the implemented
             factorisation must move (DESIGN.md section 5) over the live kernel time and the measured peak,
             `frac_pipe_measured` = ncu's shared-memory wavefronts of the committed profile x 128 B over the same,
             `survey_model` = SURVEY 8(d)'s 4-pass byte model (can exceed 1: the kernels move less than it charges)
  cpu_baseline  BASELINE.md rows B1 (literal search.cpp, one core) and B2 (forked over all cores) plus the OpenMP
             oracle port, on a bounded sample of the same captures (N = 1, rank 0)
`--impl reference` times the reference's own CPU path on the same workload instead (see reference_arm()).
`--dump-outputs DIR` writes the records the last timed step of each workload returned (dump_records()); the inputs are
generated from fixed seeds, so two builds run with the same arguments can be compared record for record.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "acquisition cells/sec (PRN x Doppler x code-phase)"
UNIT = "cells/s"
HEADLINE = "cfg5"
CAPTURES_TOTAL = 1024
# SURVEY.md 8(d): algorithmic work per tile (one inverse FFT of one (sat, Doppler, block))
FLOP_PER_TILE = {4092: 6 * 16384 + 5 * 16384 * 14 + 3 * 4092, 16368: 6 * 16384 + 5 * 16384 * 14 + 3 * 16368}
SMEM_BYTES_PER_TILE = {4092: 131072 + 1048576 + 4092 * 8, 16368: 131072 + 1048576 + 16368 * 8}
L2_NOTE = "256 MiB flush write between timed steps, outside the event pairs"


def log(*a):
    print(*a, file=sys.stderr, flush=True)


# ------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed regions (B200_PROFILING.md recipe).
    nvidia-smi needs a few hundred ms to deliver its first sample: it is started before the first warm-up, samples
    carry timestamps, and a region reports the samples between its own start and end marks."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap,timestamp")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.rows = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None

    @staticmethod
    def _epoch(stamp):
        import datetime
        try:
            return datetime.datetime.strptime(stamp, "%Y/%m/%d %H:%M:%S.%f").timestamp()
        except ValueError:
            return None

    def stop(self):
        if not self.proc:
            self.rows = []
            return
        time.sleep(0.05)
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
            out, _ = self.proc.communicate()
        rows = []
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                row = (float(f[1]), float(f[2]), float(f[3]))
            except ValueError:
                continue
            rs = {name for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], f[5:9])
                  if v.lower().startswith("active")}
            rows.append((self._epoch(f[9]) if len(f) > 9 else None, row, rs))
        self.rows = rows

    def region(self, t0, t1):
        """Clock summary over [t0, t1] (time.time() stamps); a region shorter than the sampling period falls back to
        every sample of the run and says so."""
        rows = self.rows or []
        if not rows:
            return None
        inside = [r for r in rows if r[0] is not None and t0 <= r[0] <= t1]
        use = inside or rows
        reasons = set().union(*[r[2] for r in use])
        return {"sm_mhz": statistics.median([r[1][0] for r in use]), "sm_max_mhz": max(r[1][1] for r in use),
                "power_w": statistics.median([r[1][2] for r in use]),
                "reasons": sorted(reasons), "samples": len(use), "samples_in_timed_region": len(inside),
                "samples_total": len(rows), "period_ms": 20}


def dump_records(out_dir, name, rec):
    """One workload's records as DIR/<name>_<field>.npy, float64 (exact for every field: int32 and float32)."""
    os.makedirs(out_dir, exist_ok=True)
    for f in rec.dtype.names:
        np.save(os.path.join(out_dir, "%s_%s.npy" % (name, f)), np.ascontiguousarray(rec[f], np.float64))


# ------------------------------------------------------------------------------------------ workload description
def config_dict(cfg, n_gpus):
    """The `config` object of the JSON line: the workload only, identical for both arms."""
    from flydog_sdr_gps_b200 import scenarios
    table = scenarios.table(cfg)
    kw = scenarios.params_kw(cfg)
    n_dop = kw.get("dop_hi", 20) - kw.get("dop_lo", -20) + 1
    k = kw.get("k_noncoh", 1)
    n_cap = CAPTURES_TOTAL if cfg == "cfg5" else 1
    cells = sum(n_dop * (16368 if r[3] == 3 else 4092) for r in table) * n_cap
    return {"workload": cfg, "detail": scenarios.CONFIGS[cfg], "captures_total": n_cap, "sats": len(table),
            "doppler_indices": n_dop, "k_noncoh": k, "cells_per_step": cells, "tiles_per_step": len(table) * n_dop * k * n_cap,
            "n_gpus": n_gpus,
            "sharding": ("%d captures sharded over %d ranks (strong scaling), records gathered" % (n_cap, n_gpus))
            if cfg == "cfg5" else ("satellite list sharded over %d ranks, capture given to every rank" % n_gpus
                                   if n_gpus > 1 else "single GPU"),
            "l2": L2_NOTE}


def farm_signals(c):
    from flydog_sdr_gps_b200 import scenarios
    return scenarios.signals("cfg5", c)


def farm_captures_numpy(idx):
    """Receiver-farm captures by index, numpy generator (CPU arms and small samples)."""
    from flydog_sdr_gps_b200 import scenarios, synth
    table = scenarios.table("cfg5")
    return np.stack([synth.make_capture(77_000 + c, 1, table, farm_signals(c)) for c in idx])


def single_capture(cfg):
    from flydog_sdr_gps_b200 import scenarios, synth
    table = scenarios.table(cfg)
    kw = scenarios.params_kw(cfg)
    return synth.make_capture(10_000 + int(cfg[3]) + len(cfg), kw.get("k_noncoh", 1), table, scenarios.signals(cfg, int(cfg[3])))


# ------------------------------------------------------------------------------------------ CPU baselines
_ref_pool_caps = None


def _ref_worker(args):
    cap_idx, sats = args
    from oracle import oracle_py as O
    t0 = time.perf_counter()
    O.ref_search(_ref_pool_caps[cap_idx], np.asarray(sats, np.int32), lib=O.ref_bench())
    return time.perf_counter() - t0


class LiteralReference:
    """The UNMODIFIED gps/search.cpp (oracle/_ref: Sample() + Correlate() per satellite, serial over the satellites
    like SearchTask, gps/search.cpp:530-602), forked over host cores -- processes, not threads: the reference keeps its
    buffers in file statics (gps/search.cpp:51-58,97).  FFT provider: the in-repo fp32 FFT (FFTW is not installed).
    Timed build: the reference's own optimisation level, -Ofast, with AVX2/FMA (oracle/_ref/libref_search_ofast.so; 2.8x
    the strict parity build, identical decisions) where the host can run it -- `self.build` says which."""

    def __init__(self, captures, n_procs):
        global _ref_pool_caps
        import multiprocessing as mp
        from oracle import oracle_py as O
        O.ref_bench()  # SearchInit once, inherited by fork
        self.build = O.REF_BENCH_BUILD
        _ref_pool_caps = captures
        self.n = n_procs
        self.pool = mp.get_context("fork").Pool(n_procs) if n_procs > 1 else None
        self.captures = captures

    def run(self, jobs):
        """jobs: list of (capture index, sat list).  Returns wall seconds."""
        t0 = time.perf_counter()
        if self.pool:
            self.pool.map(_ref_worker, jobs, chunksize=1)
        else:
            for j in jobs:
                _ref_worker(j)
        return time.perf_counter() - t0

    def close(self):
        if self.pool:
            self.pool.close()
            self.pool.join()


def fftw_probe():
    """SURVEY 8(d): the CPU rows use FFTW if the box has it.  Record the attempt."""
    import ctypes
    for name in ("libfftw3f.so.3", "libfftw3f.so"):
        try:
            ctypes.CDLL(name)
            return {"library": name, "available": True,
                    "used": False, "note": "present, but oracle/_ref was built against the in-repo FFT shim"}
        except OSError as e:
            err = str(e)
    return {"library": "libfftw3f.so.3", "available": False, "error": err,
            "note": "rows are search.cpp + in-repo fp32 FFT (FFTW unavailable)"}


def cpu_baseline_rows(cells_per_sat=41 * 4092, target_s=4.0):
    """BASELINE.md section 3 on this box's host cores, bounded samples of the cfg5 captures (identical bytes as the GPU
    arm's generator family): each row is sized from a short probe to about `target_s` seconds of wall time."""
    from oracle import oracle_py as O
    from flydog_sdr_gps_b200 import scenarios
    cores = os.cpu_count() or 1
    table = scenarios.table("cfg5")
    out = {"fftw": fftw_probe(), "rows": {}}
    O.build(ref=False)
    caps = farm_captures_numpy(range(max(2, cores)))
    sats32 = list(range(32))
    if O.have_ref():
        lit1 = LiteralReference(caps, 1)
        lit1.run([(0, [0])])  # page-in
        probe = lit1.run([(0, sats32[:8])]) / 8                       # seconds per satellite on one core
        n1 = max(1, min(64, int(target_s / (32 * probe))))            # whole captures
        dt = lit1.run([(c % len(caps), sats32) for c in range(n1)])
        out["build"] = lit1.build
        out["rows"]["B1_literal_search_cpp_1core"] = {
            "value": n1 * 32 * cells_per_sat / dt, "unit": UNIT, "cores": 1, "ms_per_sat": dt / (n1 * 32) * 1e3,
            "sample": "%d cfg5 captures x 32 Navstar PRNs, Sample()+Correlate() per sat, serial (%.2f s)" % (n1, dt)}
        lit = LiteralReference(caps, cores)
        lit.run([(p, [0]) for p in range(cores)])
        per = max(1, min(64, int(target_s / (32 * probe))))           # captures per process
        dt = lit.run([(p, sats32) for p in range(cores)] * per)
        out["rows"]["B2_literal_search_cpp_all_cores"] = {
            "value": per * cores * 32 * cells_per_sat / dt, "unit": UNIT, "cores": cores,
            "sample": "%d processes x %d cfg5 captures x 32 PRNs (%.2f s)" % (cores, per, dt)}
        lit.close()
    prm = O.default_params()
    O.search(caps[0], table, sel=np.arange(1, dtype=np.int32), params=prm, nthreads=1)
    t0 = time.perf_counter()
    O.search(caps[0], table, params=prm, nthreads=cores)
    probe = time.perf_counter() - t0
    reps = max(2, min(256, int(target_s / probe)))
    t0 = time.perf_counter()
    for r in range(reps):
        O.search(caps[r % len(caps)], table, params=prm, nthreads=cores)
    dt = time.perf_counter() - t0
    out["rows"]["port_oracle_openmp_all_cores"] = {
        "value": reps * 32 * cells_per_sat / dt, "unit": UNIT, "cores": min(cores, 32),
        "sample": "%d cfg5 captures x 32 PRNs, OpenMP over satellites (%.2f s)" % (reps, dt)}
    head = out["rows"].get("B2_literal_search_cpp_all_cores") or out["rows"]["port_oracle_openmp_all_cores"]
    out.update({"value": head["value"], "unit": UNIT, "cores": head["cores"],
                "kind": "reference" if "B2_literal_search_cpp_all_cores" in out["rows"] else "port",
                "sample": head["sample"] + "; FFT = in-repo fp32 FFT behind the FFTW API (FFTW unavailable); build " +
                str(out.get("build", "-O2 strict (oracle port)"))})
    return out


# ------------------------------------------------------------------------------------------ reference arm
def reference_arm(args):
    """--impl reference: the reference's own CPU implementation of the path on this box's host cores, on the headline
    workload.  cfg5 is the reference's own search (32 Navstar PRNs, bins -20..+20, K = 1), so the timed code is the
    UNMODIFIED gps/search.cpp (oracle/_ref), one process per core, each searching whole captures satellite by satellite
    like SearchTask; each step is a bounded sample of the 1024 captures (one per core).  Without oracle/_ref (reference
    tree absent at build time) the OpenMP oracle port runs instead and the line says so."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from oracle import oracle_py as O
    from flydog_sdr_gps_b200 import scenarios
    O.build(ref=False)
    cores = os.cpu_count() or 1
    table = scenarios.table(HEADLINE)
    steps, warm = args.steps, args.warmup
    caps = farm_captures_numpy(range(cores))
    cells_cap = 32 * 41 * 4092
    if O.have_ref():
        kind = "reference"
        lit = LiteralReference(caps, cores)
        build = lit.build
        one = [(p, list(range(32))) for p in range(cores)]
        probe = lit.run(one)                                   # one capture per core
        per = max(1, min(16, int(1.0 / max(probe, 1e-3))))     # captures per core and step: about a second per step
        jobs = one * per
        sample = "each step: %d of the %d captures (%d per core) x 32 PRNs x 41 bins, unmodified gps/search.cpp forked over %d processes" % (
            per * cores, CAPTURES_TOTAL, per, cores)
        for _ in range(min(warm, 1)):
            lit.run(jobs)
        dts = [lit.run(jobs) for _ in range(steps)]
        lit.close()
        n_caps_step = per * cores
    else:
        kind = "port"
        build = "-O2 strict IEEE (oracle port)"
        prm = O.default_params()
        n_caps_step = 2
        sample = "each step: 2 of the %d captures x 32 PRNs x 41 bins, OpenMP oracle port (oracle/_ref not built)" % CAPTURES_TOTAL
        for _ in range(min(warm, 1)):
            O.search(caps[0], table, params=prm, nthreads=cores)
        dts = []
        for _ in range(steps):
            t0 = time.perf_counter()
            for c in range(n_caps_step):
                O.search(caps[c % len(caps)], table, params=prm, nthreads=cores)
            dts.append(time.perf_counter() - t0)
    dt = sum(dts) / len(dts)
    value = n_caps_step * cells_cap / dt
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
            "warmup": warm, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": config_dict(HEADLINE, args.gpus),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind,
                             "sample": sample + "; FFT = in-repo fp32 FFT behind the FFTW API (FFTW unavailable); build " + build,
                             "build": build, "fftw": fftw_probe()},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)
    return 0


def cufft_point(torch, batch, reps=20):
    """cuFFT through torch.fft.ifft: `batch` unnormalised 16384-point complex64 inverse transforms per call, input and
    output resident.  ONLY the transform: the engine's tile also forms the product, the power, the non-coherent sum and
    the peak search, and never writes the lags."""
    x = torch.randn(batch, 16384, dtype=torch.complex64, device="cuda")
    for _ in range(3):
        y = torch.fft.ifft(x, norm="forward")
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        y = torch.fft.ifft(x, norm="forward")
    b.record()
    torch.cuda.synchronize()
    ms = a.elapsed_time(b) / reps
    del y, x
    return {"what": "torch.fft.ifft (cuFFT) %d x 16384 complex64, out-of-place, transform only" % batch,
            "batch": batch, "ms_per_call": ms, "transforms_per_s": batch / (ms * 1e-3)}


# ------------------------------------------------------------------------------------------ our arm
class Timer:
    """Device-side and end-to-end timing of a step function pair under the contract's rules."""

    def __init__(self, torch, dist, world, flush):
        self.torch, self.dist, self.world, self.flush = torch, dist, world, flush

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, x):
        t = self.torch.tensor([x], dtype=self.torch.float64, device="cuda")
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def device(self, step, steps, warmup):
        """K steps bracketed by CUDA events on the launching stream, L2 flushed before each (outside the event pair);
        returns ms per step (max over ranks of the summed event times) and the wall-clock window."""
        torch = self.torch
        for _ in range(warmup):
            step()
        self.barrier()
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        t0 = time.time()
        for a, b in evs:
            self.flush.fill_(1)
            a.record()
            step()
            b.record()
        self.barrier()
        t1 = time.time()
        ms = sum(a.elapsed_time(b) for a, b in evs)
        return self.max_over_ranks(ms) / steps, (t0, t1)

    def wall(self, step, steps, warmup):
        """End to end: K synchronous calls, wall clock, barrier + synchronize on both sides, max over ranks."""
        for _ in range(warmup):
            step()
        self.barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            step()
        self.torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        return self.max_over_ranks(dt) / steps * 1e3


def kernel_counters():
    """ncu counters of the committed profiles, per tile (profiles/r2_kernel_counters.json; tools/ncu_summary.py)."""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "r2_kernel_counters.json")))
    except Exception:
        return {}


def algo_smem_bytes_per_tile(lag, k, half_bin):
    """Shared-memory bytes one (satellite, Doppler) tile of k blocks must move BY DESIGN in the implemented factorisation
    (DESIGN.md section 5): per 4096-point sub-FFT 32 KiB per pass of 256 threads x 16 points -- two exchanges (write +
    read each: 128 KiB), every operand that is staged in shared memory (bulk-copy write + read: 64 KiB each) and the
    15 KiB of stage-B twiddle reads where that table lives in shared memory; four sub-FFTs per block.  An operand resident
    in tensor memory (the capture residue for K = 1 on full bins, the code run for K > 1) costs nothing here."""
    kib = 1024
    if lag == 4092:
        if k > 1:      # k_search_l1_multi: D staged every block, E staged in block 0 only, twiddle table in smem
            return k * 4 * (64 + 128 + 15) * kib + 4 * 64 * kib
        if half_bin:   # k_search_l1<false>: both operands staged, twiddles in tensor memory
            return 4 * (64 + 64 + 128) * kib
        return 4 * (64 + 128 + 15) * kib   # k_search_l1_cr: E staged, D resident, twiddle table in smem
    if k > 1:          # k_search_e1b_multi: D staged, E from L2, twiddle table, 32 KiB of block powers written + read
        return k * (4 * (64 + 128 + 15) + 64) * kib
    return 4 * (64 + 64 + 128 + 15) * kib   # k_search_e1b: both operands staged, twiddle table in smem


def roofline_of(cfg, table, n_dop, k, n_cap, search_ms, step_kern_ms, mb, peaks):
    lags = [16368 if r[3] == 3 else 4092 for r in table]
    flop = sum(k * n_dop * FLOP_PER_TILE[l] for l in lags) * n_cap
    survey_b = sum(k * n_dop * SMEM_BYTES_PER_TILE[l] for l in lags) * n_cap
    smem_b = sum(n_dop * algo_smem_bytes_per_tile(l, k, cfg == "cfg2") for l in lags) * n_cap
    hbm_b = n_cap * k * 8192 + len(table) * 16384 * 8 + 24 * len(table) * n_cap
    # what the search KERNEL itself must read when its inputs are not cache-resident: the capture spectra the forward FFT
    # left behind (128 KiB per capture, block and half-bin variant) and the extended code rows (~128 KiB per satellite)
    nvar = 2 if cfg == "cfg2" else 1
    hbm_kernel_b = n_cap * k * nvar * 16384 * 8 + len(table) * 16384 * 8 + 16 * len(table) * n_dop * n_cap
    tiles = len(table) * n_dop * k * n_cap
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    sec = search_ms * 1e-3
    fp32_ach, smem_ach, hbm_ach = flop / sec / 1e12, smem_b / sec / 1e12, hbm_b / sec / 1e9
    ctr = kernel_counters().get(cfg) or {}
    r = {
        "bound": "smem",
        "kernel": ctr.get("kernel", "k_search_l1 / k_search_l1_multi / k_search_e1b (conj-multiply + 16384-pt inverse FFT + |.|^2 + peak search)"),
        "achieved": smem_ach * 1e3, "peak": mb["smem_tbs"] * 1e3, "unit": "GB/s", "frac": smem_ach / mb["smem_tbs"],
        "peak_source": "shared-memory micro-benchmark in this run (acq_microbench: conflict-free 8-byte LDS+STS); "
                       "nominal 148 SM x 128 B/clk x SM clock",
        "algorithmic_bytes_per_launch": smem_b,
        "model": "bytes the implemented factorisation must move through shared memory (DESIGN.md section 5: per 4096-point "
                 "sub-FFT two exchanges + every smem-staged operand + the stage-B twiddle table; %d B per tile of the "
                 "dominant kernel) x tiles / live kernel time / measured shared-memory peak" % algo_smem_bytes_per_tile(max(lags), k, cfg == "cfg2"),
        "survey_model": {"bytes_per_tile": SMEM_BYTES_PER_TILE[max(lags)], "bytes_per_launch": survey_b,
                         "achieved": survey_b / sec / 1e9, "frac": survey_b / sec / 1e12 / mb["smem_tbs"],
                         "note": "SURVEY 8(d)'s 4-pass model of an unfused 16384-point transform. The kernels move fewer bytes "
                                 "than it charges (three exchanges instead of four passes, pruned output, one operand and the "
                                 "parked values through tensor memory), so this fraction can exceed 1: it measures the "
                                 "algorithmic saving, not the pipe"},
        "frac_note": "frac = bytes of the implemented factorisation / kernel time / measured shared-memory peak; "
                     "frac_pipe_measured = what the L1/shared pipe physically carried (ncu wavefronts of the committed profile "
                     "x 128 B, incl. bulk-copy arbitration) over the same time and peak; fp32.frac = the FP32 lanes",
        "kernel_ms": search_ms, "kernel_share_of_step": search_ms / step_kern_ms if step_kern_ms else None,
        "traffic": ctr.get("dram_bytes_per_tile") and ctr["dram_bytes_per_tile"] * tiles,
        "achieved_smem": smem_ach, "achieved_fp32": fp32_ach, "achieved_hbm": hbm_ach,
        "fp32": {"bound": "fp32", "achieved": fp32_ach, "peak": mb["ffma_tflops"], "unit": "TFLOP/s",
                 "frac": fp32_ach / mb["ffma_tflops"], "algorithmic_flop_per_launch": flop,
                 "peak_source": "FFMA micro-benchmark in this run; nominal 148 SM x 128 lanes x 2 x clock"},
        "hbm": {"bound": "hbm", "achieved": hbm_ach, "peak": hbm_peak, "unit": "GB/s", "frac": hbm_ach / hbm_peak,
                "peak_source": "MEASURED_PEAKS.json" if "hbm_gbs" in peaks else "fallback 6650 GB/s",
                "algorithmic_bytes_per_launch": hbm_b,
                "search_kernel_input_bytes": hbm_kernel_b,
                "note": "algorithmic_bytes_per_launch = SURVEY 8(d)'s unique bytes of the whole path (packed captures + code "
                        "spectra + records); the search kernel's own inputs are the capture spectra the forward FFT wrote "
                        "(search_kernel_input_bytes; beyond L2 for a 1024-capture farm), which `traffic` (ncu, cold caches) "
                        "should be compared with. Either way HBM carries well under 1 % of its bandwidth here."},
    }
    if ctr.get("smem_wavefronts_per_tile"):
        # what the L1/shared data pipe physically carried (ncu l1tex__data_pipe_lsu_wavefronts_mem_shared of the
        # committed profile, per tile) at 128 B per wavefront, over the live kernel time
        pipe = ctr["smem_wavefronts_per_tile"] * tiles * 128 / sec / 1e12
        r["frac_pipe_measured"] = pipe / mb["smem_tbs"]
        r["pipe_measured"] = {"smem_wavefronts_per_tile": ctr["smem_wavefronts_per_tile"], "achieved_tbs": pipe,
                              "fma_pipe_pct_ncu": ctr.get("fma_pipe_pct"), "lsu_pipe_pct_ncu": ctr.get("lsu_pipe_pct"),
                              "profile": ctr.get("profile")}
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--captures", type=int, default=CAPTURES_TOTAL, help=argparse.SUPPRESS)  # smaller farm for quick runs
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="headline only (skip the cfg1..cfg4 entries)")
    ap.add_argument("--only", default="", help="comma list of the cfg1..cfg4 entries to run (default: all)")
    ap.add_argument("--no-cufft", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the records of each workload's last timed step "
                    "as DIR/<workload>_<field>.npy (float64)")
    args = ap.parse_args()
    if args.impl == "reference":
        return reference_arm(args)
    args.warmup = max(args.warmup, 3)

    import torch
    import flydog_sdr_gps_b200 as F
    from flydog_sdr_gps_b200 import farm, scenarios, synth

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the engine has no CPU fallback")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")  # > 126 MB L2
    # a non-default stream: its handle is non-NULL, so the engine launches on exactly this stream and
    # torch.cuda.Event timing brackets the engine's kernels (NULL would select the engine's own stream)
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    T = Timer(torch, dist, world, flush)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass

    # ================================================================= headline: cfg5, 1024 captures, strong scaling
    n_total = args.captures
    table = scenarios.table(HEADLINE)
    eng = F.AcqEngine(table, F.default_params(), device=local)
    fm = farm.CaptureFarm(eng, n_total, eng.k_noncoh * eng.block_bytes, len(table), dist=dist)
    t_gen = time.time()
    idx = range(fm.lo, fm.hi)
    caps_dev = synth.make_capture_batch_torch([77_000 + c for c in idx], 1, table, [farm_signals(c) for c in idx], "cuda")
    fm.load(caps_dev.cpu().numpy())
    del caps_dev
    log("rank %d: %d captures generated in %.1f s" % (rank, fm.n_local, time.time() - t_gen))
    cells_total = eng.cells_per_search() * n_total
    tiles_total = eng.tiles_per_search() * n_total
    launches0 = eng.launch_count
    ms_per_step, window = T.device(fm.search_resident, args.steps, args.warmup)
    launches = eng.launch_count - launches0 - 0
    launches_timed = launches * args.steps // (args.steps + args.warmup)
    value = cells_total / (ms_per_step * 1e-3)
    dev_records = fm.d_all.cpu().numpy().copy()
    if args.dump_outputs and rank == 0:
        dump_records(args.dump_outputs, HEADLINE, fm._unpad(dev_records, fm.n_sel).reshape(n_total, fm.n_sel))
    # per-kernel durations (CUDA events between the kernels on the launching stream), same window of clock samples
    eng.set_profiling(True)
    kern_ms = []
    for _ in range(min(args.steps, 10)):
        flush.fill_(1)
        fm.search_resident()
        kern_ms.append(eng.kernel_ms())
    T.barrier()
    eng.set_profiling(False)
    # end to end through host buffers
    e2e_ms = T.wall(fm.search, args.steps, 3)
    rec = fm.search()
    same = bool(np.array_equal(fm.h_all.numpy(), dev_records))
    detected = int((rec["snr"] >= 16.0).sum())
    # spot check against single searches through the C ABI (bitwise)
    spot_ok = True
    if fm.n_local:
        one = eng.search(fm.h_in.numpy()[:8192])
        spot_ok = bool(one[0].tobytes() == rec[fm.lo].tobytes())
    t_end_head = time.time()

    search_ms = statistics.mean(k["search"] for k in kern_ms)
    step_kern_ms = statistics.mean(sum(k.values()) for k in kern_ms)
    mb = F.microbench(local)

    # ================================================================= cfg1..cfg4
    entries = {}
    todo = [] if args.no_configs else [c for c in ("cfg1", "cfg2", "cfg3", "cfg4", "cfg3_k4") if not args.only or c in args.only.split(",")]
    for cfg in todo:
        tb = scenarios.table(cfg)
        kw = scenarios.params_kw(cfg)
        e = eng if cfg == "cfg1" else F.AcqEngine(tb, F.default_params(**kw), device=local)
        cap = single_capture(cfg)
        steps_c = args.steps
        cells_c, tiles_c = e.cells_per_search(), e.tiles_per_search()
        ent = {"cells_per_step": cells_c, "tiles_per_step": tiles_c, "steps": steps_c}
        if world == 1:
            d_in = torch.from_numpy(cap).cuda()
            d_out = torch.zeros(len(tb) * 24, dtype=torch.uint8, device="cuda")
            h_in = torch.from_numpy(cap).pin_memory()
            h_out = torch.zeros(len(tb) * 24, dtype=torch.uint8).pin_memory()
            l0 = e.launch_count
            ms, win = T.device(lambda: e.search_device(d_in.data_ptr(), d_out.data_ptr(), 1, stream_ptr=stream.cuda_stream),
                               steps_c, args.warmup)
            ent["gpu_launches_per_step"] = (e.launch_count - l0) // (steps_c + args.warmup)
            e2 = T.wall(lambda: e.search_ptr(h_in.data_ptr(), 1, h_out.data_ptr()), steps_c, 3)
            ent["device_equals_host_path"] = bool(torch.equal(d_out.cpu(), h_out))
            ent["e2e"] = {"value": cells_c / (e2 * 1e-3), "unit": UNIT, "ms_per_step": e2, "h2d_bytes_per_step": int(cap.size),
                          "d2h_bytes_per_step": len(tb) * 24,
                          "api": "acq_search (C ABI, host buffers)" + (
                              ": the 8 KiB capture travels host -> device as the front-end kernel's argument, the records "
                              "come back through mapped pinned memory" if cap.size == 8192 else
                              ": pinned staging + H2D copy node, records through mapped pinned memory")}
            ent["sharding"] = "single GPU"
            e.set_profiling(True)
            km = []
            for _ in range(min(steps_c, 10)):
                flush.fill_(1)
                e.search_device(d_in.data_ptr(), d_out.data_ptr(), 1, stream_ptr=stream.cuda_stream)
                km.append(e.kernel_ms())
            e.set_profiling(False)
            nrec = h_out.numpy().view(F.RECORD_DTYPE)
        else:
            sf = farm.SatFarm(e, len(tb), cap.size, dist=dist)
            sf.load(cap)
            ms, win = T.device(sf.search_resident, steps_c, args.warmup)
            e2 = T.wall(sf.search, steps_c, 3)
            nrec = sf.search().copy()
            ent["e2e"] = {"value": cells_c / (e2 * 1e-3), "unit": UNIT, "ms_per_step": e2, "h2d_bytes_per_step": sf.h2d_bytes,
                          "d2h_bytes_per_step": sf.d2h_bytes,
                          "api": "farm.SatFarm.search: H2D of the capture on every rank, acq_search_device on a slice of "
                                 "the table, NCCL all_gather of the records, D2H"}
            ent["sharding"] = "satellite list split over %d ranks (%d..%d per rank), capture given to every rank; " \
                              "latency-bound: launch + NCCL gather of 24-byte records (SURVEY 8(e))" % (
                                  world, min(sf.counts), max(sf.counts))
            e.set_profiling(True)
            km = []
            for _ in range(min(steps_c, 10)):
                flush.fill_(1)
                sf.search_resident()
                km.append(e.kernel_ms())
            T.barrier()
            e.set_profiling(False)
        if args.dump_outputs and rank == 0:
            dump_records(args.dump_outputs, cfg, nrec)
        thr = kw.get("thr_e1b", 16.0) if cfg.startswith("cfg3") else kw.get("thr_l1", 16.0)
        ent.update({"value": cells_c / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "tiles_per_s": tiles_c / (ms * 1e-3),
                    "kernel_ms": {k: statistics.mean(x[k] for x in km) for k in km[0]},
                    "detected": int((nrec["snr"] >= thr).sum()), "window": win})
        if rank == 0:
            sm = statistics.mean(x["search"] for x in km)
            n_cap_shard = 1
            tb_local = tb if world == 1 else tb[scenarios.shard(len(tb), 0, world)[0]:scenarios.shard(len(tb), 0, world)[1]]
            rf = roofline_of(cfg, tb_local, e.n_dop, e.k_noncoh, n_cap_shard, sm, statistics.mean(sum(x.values()) for x in km), mb, peaks)
            ent["roofline"] = {"frac": rf["frac"], "frac_fp32": rf["fp32"]["frac"], "kernel_ms": sm,
                               "frac_pipe_measured": rf.get("frac_pipe_measured"), "bound": "smem",
                               "frac_survey_model": rf["survey_model"]["frac"],
                               "note": "search kernel(s) of rank 0's share"}
        entries[cfg] = ent
        if e is not eng:
            e.close()
    if world > 1 and "cfg4" in entries:
        entries["cfg4_prn_sharded"] = dict(entries["cfg4"], what="BASELINE configs[3]: 82 PRNs of one capture sharded over the ranks")

    if rank == 0:
        sampler.stop()
    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return 0

    for ent in entries.values():
        ent["clocks"] = sampler.region(*ent.pop("window"))
    share_tables = table  # every rank searches the whole table on its captures
    n_cap_rank0 = fm.n_local
    roofline = roofline_of(HEADLINE, share_tables, eng.n_dop, eng.k_noncoh, n_cap_rank0, search_ms, step_kern_ms, mb, peaks)
    roofline["microbench"] = mb
    cfgd = config_dict(HEADLINE, world)
    if n_total != CAPTURES_TOTAL:
        cfgd.update({"captures_total": n_total, "cells_per_step": cells_total, "tiles_per_step": tiles_total,
                     "note": "reduced farm (--captures): not the BASELINE size"})
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "config": cfgd,
        "tiles_per_s": tiles_total / (ms_per_step * 1e-3),
        "timed_region_s": ms_per_step * args.steps * 1e-3,
        "e2e": {"value": cells_total / (e2e_ms * 1e-3), "unit": UNIT, "ms_per_step": e2e_ms,
                "h2d_bytes_per_step": fm.h2d_bytes * world if world == 1 else n_total * 8192,
                "d2h_bytes_per_step": fm.d2h_bytes * world,
                "api": "farm.CaptureFarm.search: pinned captures -> H2D -> acq_search_device -> NCCL all_gather of the "
                       "records -> D2H of all %d records on every rank" % (n_total * len(table))},
        "gpu_launches": int(launches_timed),
        "kernel_ms": {k: statistics.mean(x[k] for x in kern_ms) for k in kern_ms[0]},
        "device_equals_host_path": same and spot_ok,
        "detected_sats": detected,
        "clocks": sampler.region(*window),
        "roofline": roofline,
        "configs": entries,
    }
    if not args.no_cufft:
        line["cufft_comparison"] = [cufft_point(torch, 4096), cufft_point(torch, 256)]
    if world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline_rows()
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
