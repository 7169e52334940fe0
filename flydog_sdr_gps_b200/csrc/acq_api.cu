// acq_api.cu -- the C ABI of include/acq_b200.h: engine lifetime, device memory, launch sequencing.
// No CPU fallback exists: every entry point either runs the sm_100a kernels or returns an error.
#include <cuda_runtime.h>

#include <cmath>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include <algorithm>
#include <cstdarg>
#include <memory>
#include <numeric>

#include "acq_geom.h"
#include "acq_kernels.cuh"

namespace {

thread_local std::string g_err;

int fail(int code, const char *fmt, ...) __attribute__((format(printf, 2, 3)));
int fail(int code, const char *fmt, ...)
{
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}

#define CU(call)                                                                                          \
    do {                                                                                                  \
        cudaError_t _e = (call);                                                                          \
        if (_e != cudaSuccess)                                                                            \
            return fail(ACQ_ERR_CUDA, "%s:%d %s: %s", __FILE__, __LINE__, #call, cudaGetErrorString(_e)); \
    } while (0)

// Restores the caller's current device on scope exit (the host application may own other GPUs).
struct DeviceGuard {
    int prev = -1;
    explicit DeviceGuard(int dev)
    {
        if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
        if (prev != dev) cudaSetDevice(dev);
        else prev = -1;
    }
    ~DeviceGuard()
    {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

// Galileo E1-B primary codes, packed (Galileo OS SIS ICD Annex C; see tools/gen_e1b_table.py).
const uint32_t kE1bWords[50 * 128] = {
#include "e1b_codes.inc"
};

// GPS C/A code (IS-GPS-200): G1 = 1 + x^3 + x^10, G2 = 1 + x^2 + x^3 + x^6 + x^8 + x^9 + x^10, both preset
// to all ones; chip = G1[10] ^ G2[t1] ^ G2[t2].  QZSS/SBAS rows of the satellite table give the G2 preset
// instead of taps (t1 or t2 > 10): chip = G1[10] ^ G2[10] with bit (i-1) of t2 loaded into stage i.
// Same conventions as the reference's CACODE (gps/cacode.h:23-64).  Packs 1023 chips LSB-first.
void ca_code_bits(int t1, int t2, uint32_t *words)
{
    const bool preset = (t1 > 10 || t2 > 10);
    int g1[11], g2[11];
    for (int i = 1; i <= 10; i++) {
        g1[i] = 1;
        g2[i] = preset ? ((t2 >> (i - 1)) & 1) : 1;
    }
    memset(words, 0, 128 * sizeof(uint32_t));
    for (int n = 0; n < 1023; n++) {
        const int chip = preset ? (g1[10] ^ g2[10]) : (g1[10] ^ g2[t1] ^ g2[t2]);
        words[n >> 5] |= (uint32_t)chip << (n & 31);
        const int f1 = g1[3] ^ g1[10];
        const int f2 = g2[2] ^ g2[3] ^ g2[6] ^ g2[8] ^ g2[9] ^ g2[10];
        for (int i = 10; i > 1; i--) {
            g1[i] = g1[i - 1];
            g2[i] = g2[i - 1];
        }
        g1[1] = f1;
        g2[1] = f2;
    }
}

using namespace acq;

// Owner of device memory, freed with the owner.  alloc() replaces the contents by n uninitialised elements.
template <typename T>
struct DevBuf {
    T *p = nullptr;
    size_t cap = 0;   // elements; 0 while p is NULL
    DevBuf() = default;
    DevBuf(const DevBuf &) = delete;
    DevBuf &operator=(const DevBuf &) = delete;
    ~DevBuf() { reset(); }
    operator T *() const { return p; }
    void reset()
    {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
    cudaError_t alloc(size_t n)
    {
        reset();
        const cudaError_t ce = cudaMalloc(&p, n * sizeof(T));
        if (ce == cudaSuccess) cap = n;
        return ce;
    }
};

// Owner of pinned host memory (cudaHostAlloc with Flags); mapped memory is zeroed and its device address kept in dev.
template <typename T, unsigned Flags>
struct PinnedBuf {
    T *p = nullptr, *dev = nullptr;
    size_t cap = 0;
    PinnedBuf() = default;
    PinnedBuf(const PinnedBuf &) = delete;
    PinnedBuf &operator=(const PinnedBuf &) = delete;
    ~PinnedBuf() { reset(); }
    void reset()
    {
        if (p) cudaFreeHost(p);
        p = dev = nullptr;
        cap = 0;
    }
    cudaError_t alloc(size_t n)
    {
        reset();
        cudaError_t ce = cudaHostAlloc(&p, n * sizeof(T), Flags);
        if (ce == cudaSuccess && (Flags & cudaHostAllocMapped)) {
            memset(p, 0, n * sizeof(T));
            ce = cudaHostGetDevicePointer(&dev, p, 0);
        }
        if (ce == cudaSuccess) cap = n;
        return ce;
    }
};

// b = a device copy of v (left empty if the copy fails)
template <typename T>
cudaError_t upload(DevBuf<T> &b, const std::vector<T> &v)
{
    cudaError_t ce = b.alloc(v.size());
    if (ce == cudaSuccess && (ce = cudaMemcpy(b.p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice)) != cudaSuccess)
        b.reset();
    return ce;
}

// Rows first..F-1 of the sub-bin rotation table [F][16384]: row v = exp(-2 pi i (v / F) n / N), double precision rounded
// once.  The angle is pi (a n) / (b N) with a / b = 2 v / F in lowest terms, so that the row v = F / 2 of an even F is
// formed by the same operations as the half-bin table (F = 2, row 1: pi n / N) and rounds to the same floats.
std::vector<float2> rotation_table(int F, int first)
{
    const double pi = 3.14159265358979323846264338327950288;
    std::vector<float2> rot((size_t)(F - first) * kN);
    for (int v = first; v < F; v++) {
        const int g = std::gcd(2 * v, F), a = 2 * v / g, b = F / g;
        for (int n = 0; n < kN; n++) {
            const double ang = pi * (double)((long long)a * n) / (double)((long long)b * kN);
            rot[(size_t)(v - first) * kN + n] = make_float2((float)cos(ang), (float)(-sin(ang)));
        }
    }
    return rot;
}

}  // namespace

struct acq_engine {
    int device = 0, sm_count = 0, sm_clock_khz = 0;
    acq_params prm{};
    std::vector<acq_sat> sats;
    int n_dop = 0, nvar = 1, Q = 0, ext_len = 0;
    int n_shift = 1, smax = 0, cd_div = 385;  // code-Doppler compensation: shifted copies per spectrum (1 = off)
    int sample_bits = 1;       // capture format: 1 = sign only (reference), 2 = sign plane + magnitude plane
    size_t block_bytes = ACQ_BLOCK_BYTES;
    cudaStream_t stream = nullptr;
    cudaEvent_t done = nullptr;
    bool pending = false;       // acq_submit outstanding
    int pending_rows = 0;       // ... whose records still sit in h_records (copied to pending_out by acq_poll/acq_wait)
    acq_record *pending_out = nullptr;
    // device-path ordering: an event behind the last device-path work on another stream; whatever touches the shared
    // scratch next waits for it (wait_scratch / hold_scratch)
    cudaEvent_t dev_done = nullptr;
    bool dev_pending = false;
    int64_t launches = 0;
    bool profiling = false, prof_valid = false;
    cudaEvent_t prof[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};

    // persistent device data
    DevBuf<float2> d_tables, d_rot, d_C, d_Ep;
    // per-call scratch (grown on demand)
    DevBuf<uint8_t> d_packed;
    DevBuf<float2> d_x2, d_Dp;   // [spectrum rows][kN] each
    DevBuf<acq_cell> d_cells;
    DevBuf<acq_record> d_records;
    DevBuf<unsigned> d_tile_ctr;    // [4] claim counters [0,1] and done counters [2,3] of the C/A and the E1B search launch (SearchArgs::tile_ctr); zero between launches
    DevBuf<unsigned> d_ctas_done;   // finished search CTAs of a small search (folded best-Doppler pick); zero between searches
    unsigned epoch = 0;             // search counter: value of the completion word
    // host path: pinned staging of small captures; records and the completion word in mapped pinned memory,
    // written by the search kernels themselves.  h_records is sized for the tagged form a polling host reads (32 B);
    // the plain 24-byte form fits too.
    PinnedBuf<uint8_t, cudaHostAllocDefault> h_packed;
    PinnedBuf<acq_record_tagged, cudaHostAllocMapped> h_records;
    PinnedBuf<unsigned, cudaHostAllocMapped> h_flag;
    // selection: work list [n_slots] (C/A entries first, then E1B) and slot -> table index
    std::vector<int32_t> sel_cache;
    int sel_kind = -1;  // -1 none, 0 whole table, 1 one satellite, 2 uploaded list
    int n_l1 = 0, n_e1b = 0, n_slots = 0;
    const int2 *cur_work = nullptr;
    const int *cur_slot_sat = nullptr;
    DevBuf<int2> d_work_full, d_work_single, d_work;   // whole table / (s, 0) per s / uploaded
    DevBuf<int> d_sat_full, d_slot_sat;                // identity / uploaded
    int full_n_l1 = 0;
    // refinement and profile: satellite types on the device, record/output scratch of the host forms (acq_profile's lag
    // profiles get a buffer per call)
    DevBuf<int> d_sat_type;
    DevBuf<acq_record> d_ref_rec;
    DevBuf<acq_fine> d_fine;
    DevBuf<acq_peak2> d_peak2;
    // The most recent search whose spectra are still on the device (captures 0: none), which refinement and profile read:
    // its slots, device slot -> satellite map and C/A and E1B slot counts.  host: a host-path search, whose records
    // acq_refine and acq_profile may take (the current selection is then its selection).  A coherent search leaves none
    // there: its shape goes to last_coh (m_coh > 0), which only acq_refine_coherent* and acq_profile_coherent* read.  A
    // search clears both when it starts.
    struct LastSearch {
        int captures = 0, slots = 0, n_l1 = 0, n_e1b = 0;
        const int *slot_sat = nullptr;
        bool host = false;
        int m_coh = 0;   // coherent: M; the spectra hold F = M (1 + half_bin) variants per block
    } last, last_coh;
    // aided host search (acq_search_aided): Doppler centres staged in pinned memory, copied to the device with the capture
    PinnedBuf<int32_t, cudaHostAllocDefault> h_center;
    DevBuf<int> d_center;
    // coherent search (acq_search_coherent): sub-bin rotation table [F][16384] of each m_coh, built on first use
    DevBuf<float2> d_rot_coh[ACQ_COH_MAX + 1];

    // Runs under the engine's device (acq_destroy, acq_create): the work in flight ends before the members free their memory.
    ~acq_engine()
    {
        if (stream) cudaStreamSynchronize(stream);
        if (dev_pending && dev_done) cudaEventSynchronize(dev_done);
        for (cudaEvent_t ev : prof)
            if (ev) cudaEventDestroy(ev);
        if (done) cudaEventDestroy(done);
        if (dev_done) cudaEventDestroy(dev_done);
        if (stream) cudaStreamDestroy(stream);
    }
};

namespace {

// What one search call asks for: the engine's whole Doppler range or, aided, a window of W = 2 half_width + 1 cells around
// each row's centre; non-coherent sums or, coherent, groups of M = m_coh blocks on the 1/F-bin grid.
struct SearchMode {
    bool aided, coherent;
    const int32_t *center;   // aided: one Doppler centre per row (host or device memory, as the entry point)
    int half_width, m_coh;
    int dop_scale() const { return coherent ? m_coh : 1; }   // dop_lo / dop_hi of the grid searched, in its units
    int variants(const acq_engine *e) const { return coherent ? m_coh * (1 + e->prm.half_bin) : e->nvar; }   // per block
    int full_dops(const acq_engine *e) const { return dop_scale() * (e->n_dop - 1) + 1; }   // n_dop, or n_dop_c
    int dops(const acq_engine *e) const { return aided ? 2 * half_width + 1 : full_dops(e); }   // cells per row
};
constexpr SearchMode kFullRange{false, false, nullptr, 0, 0};

// Build-time switch of an experiment variant (tools/build_variants.py); the product library defines none and reads no
// environment variable.
//   ACQ_ARG_INPUT=1|0        a search of ONE 1-bit block: the capture travels as the front end's kernel argument (1) or by
//                            the staging buffer and a copy node like every other search (0, variant "argin0")
#ifndef ACQ_ARG_INPUT
#define ACQ_ARG_INPUT 1
#endif
// Host path, small searches: the capture goes through an engine-owned pinned staging buffer (a pageable source would
// make cudaMemcpyAsync synchronous), the kernels write the records straight into mapped pinned memory, and the host
// polls a completion word there instead of waiting for the stream.  Above these sizes: plain copies and a stream wait.
constexpr size_t kStagePackedMax = 256u << 10;  // bytes
constexpr int kHostRecordRowsMax = 256;          // records (24 B each: single PCIe writes from the SMs)
// Up to this many (capture, sat) rows the best-Doppler pick is one CTA that polls the search CTAs' completion counter
// (k_pick_small: no wait for the grids to drain; a few microseconds at most); above, k_best_dop follows the search the
// ordinary way (nothing against a long search).
constexpr int kFoldPickRowsMax = acq::kPickSmallRowsMax;
static_assert(kHostRecordRowsMax <= kFoldPickRowsMax, "the completion word is raised by k_pick_small");

// Everything that is about to touch the shared scratch from the host (reallocation, synchronous copies) first
// drains the engine stream and the last device-path work.
int drain(acq_engine *e)
{
    CU(cudaStreamSynchronize(e->stream));
    if (e->dev_pending) {
        CU(cudaEventSynchronize(e->dev_done));
        e->dev_pending = false;
    }
    return ACQ_OK;
}

// b holds at least `need` elements: only a buffer that grows drains the engine first
template <class Buf>
int grow(acq_engine *e, Buf &b, size_t need)
{
    if (need <= b.cap) return ACQ_OK;
    int rc = drain(e);
    if (rc) return rc;
    CU(b.alloc(need));
    return ACQ_OK;
}

// Device-path ordering.  Work about to use the engine's scratch on `st` waits for the last device-path work on another
// stream (a no-op on the stream that recorded it) and, with engine_too, for what the engine stream has queued ...
int wait_scratch(acq_engine *e, cudaStream_t st, bool engine_too)
{
    if (e->dev_pending) CU(cudaStreamWaitEvent(st, e->dev_done, 0));
    if (engine_too && st != e->stream) {
        CU(cudaEventRecord(e->dev_done, e->stream));
        CU(cudaStreamWaitEvent(st, e->dev_done, 0));
    }
    return ACQ_OK;
}

// ... and once it is enqueued on a stream other than the engine's, whatever uses the scratch next (any stream, or the
// host) waits for it.
int hold_scratch(acq_engine *e, cudaStream_t st)
{
    if (st != e->stream) {
        CU(cudaEventRecord(e->dev_done, st));
        e->dev_pending = true;
    }
    return ACQ_OK;
}

// Scratch of a search of n_captures over the current selection in mode m; host_path: also the staging and record buffers
int ensure_scratch(acq_engine *e, int n_captures, bool host_path, const SearchMode &m)
{
    const size_t blocks = (size_t)n_captures * e->prm.k_noncoh;
    const size_t spectra = blocks * m.variants(e) * e->n_shift * kN;   // x2 and the capture spectra
    if (spectra > e->d_x2.cap || spectra > e->d_Dp.cap) {
        int rc = drain(e);  // changing scratch under an in-flight search is not allowed
        if (rc) return rc;
        CU(e->d_x2.alloc(spectra));
        CU(e->d_Dp.alloc(spectra));
    }
    if (m.coherent && !e->d_rot_coh[m.m_coh]) CU(upload(e->d_rot_coh[m.m_coh], rotation_table(m.variants(e), 0)));
    const size_t rows = (size_t)n_captures * e->n_slots;
    int rc;
    if ((rc = grow(e, e->d_cells, rows * m.dops(e)))) return rc;
    if (!host_path) return ACQ_OK;
    const size_t bytes = blocks * e->block_bytes;
    if ((rc = grow(e, e->d_packed, bytes))) return rc;
    if (bytes <= kStagePackedMax && (rc = grow(e, e->h_packed, bytes))) return rc;
    if (m.aided && ((rc = grow(e, e->d_center, rows)) || (rc = grow(e, e->h_center, rows)))) return rc;
    return rows <= (size_t)kHostRecordRowsMax ? grow(e, e->h_records, rows) : grow(e, e->d_records, rows);
}

// Split the selection (checked by check_search) into the 1 ms-window (Navstar/QZSS/SBAS) and E1B work lists.  The whole
// table and single satellites (what the literal SearchTask loop asks for, one satellite per capture) use lists built at
// acq_create; any other list is uploaded, which drains the engine first.
int set_selection(acq_engine *e, const int32_t *sel, int n_sel)
{
    const int n_sats = (int)e->sats.size();
    if (!sel) {
        if (e->sel_kind != 0) {
            e->sel_cache.resize(n_sats);
            for (int i = 0; i < n_sats; i++) e->sel_cache[i] = i;
            e->sel_kind = 0;
        }
        e->cur_work = e->d_work_full;
        e->cur_slot_sat = e->d_sat_full;
        e->n_l1 = e->full_n_l1;
        e->n_e1b = n_sats - e->full_n_l1;
        e->n_slots = n_sats;
        return ACQ_OK;
    }
    if (n_sel == 1) {
        const int sat = sel[0];
        e->sel_cache.assign(1, sat);
        e->sel_kind = 1;
        e->cur_work = e->d_work_single + sat;
        e->cur_slot_sat = e->d_sat_full + sat;
        e->n_e1b = (e->sats[sat].type == ACQ_E1B) ? 1 : 0;
        e->n_l1 = 1 - e->n_e1b;
        e->n_slots = 1;
        return ACQ_OK;
    }
    if (e->sel_kind == 2 && (int)e->sel_cache.size() == n_sel && std::equal(sel, sel + n_sel, e->sel_cache.begin())) {
        e->cur_work = e->d_work;
        e->cur_slot_sat = e->d_slot_sat;
        return ACQ_OK;
    }
    std::vector<int2> work;
    work.reserve(n_sel);
    int n_l1 = 0;
    for (int pass = 0; pass < 2; pass++)
        for (int i = 0; i < n_sel; i++) {
            const bool e1b = (e->sats[sel[i]].type == ACQ_E1B);
            if ((pass == 1) != e1b) continue;
            work.push_back(make_int2(sel[i], i));
            if (!e1b) n_l1++;
        }
    int rc = drain(e);  // the lists may still be read by a search in flight; the copies below are synchronous
    if (rc) return rc;
    e->sel_kind = -1;
    if ((size_t)n_sel > e->d_work.cap || (size_t)n_sel > e->d_slot_sat.cap) {
        CU(e->d_work.alloc(n_sel));
        CU(e->d_slot_sat.alloc(n_sel));
    }
    CU(cudaMemcpy(e->d_work, work.data(), work.size() * sizeof(int2), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(e->d_slot_sat, sel, (size_t)n_sel * sizeof(int), cudaMemcpyHostToDevice));
    e->sel_cache.assign(sel, sel + n_sel);
    e->sel_kind = 2;
    e->cur_work = e->d_work;
    e->cur_slot_sat = e->d_slot_sat;
    e->n_l1 = n_l1;
    e->n_e1b = n_sel - n_l1;
    e->n_slots = n_sel;
    return ACQ_OK;
}

// Largest Doppler range an engine can have: |index| <= 4094 half-bins (acq_create: at most 2048 bins either side).
constexpr int kMaxHalfWidth = 4094;

// The checks of one search call, before anything touches the device.  Those that need no engine come first, so that they
// are reported whatever the engine.  ACQ_ERR_ARG for the argument errors; ACQ_ERR_UNSUPPORTED for what the coherent
// search does not cover (E1B rows, code-Doppler engines, more than 2^24 capture spectra) and for searches above the tile
// bound: a search kernel launch indexes its tiles with 32 bits (and four units per tile with 64).
int check_search(acq_engine *e, const SearchMode &m, const void *packed, int n_captures, const int32_t *sel, int n_sel,
                 const void *out, bool device)
{
    const int hw = m.half_width;
    if (m.aided && !m.center) return fail(ACQ_ERR_ARG, "dop_center is NULL");
    if (m.aided && hw < 0) return fail(ACQ_ERR_ARG, "half_width must be >= 0 (got %d)", hw);
    if (m.coherent && (m.m_coh < 1 || m.m_coh > ACQ_COH_MAX))
        return fail(ACQ_ERR_ARG, "m_coh=%d outside 1..%d", m.m_coh, ACQ_COH_MAX);
    if (m.aided && hw > (m.coherent ? ACQ_COH_MAX : 1) * kMaxHalfWidth)
        return fail(ACQ_ERR_ARG, "Doppler window W = 2*half_width+1 with half_width %d exceeds n_dop%s of any engine", hw,
                    m.coherent ? "_c" : "");
    if (!e) return fail(ACQ_ERR_ARG, "engine is NULL");
    const int full = m.full_dops(e), K = e->prm.k_noncoh;
    if (m.aided && 2 * hw + 1 > full) {
        if (m.coherent)
            return fail(ACQ_ERR_ARG, "Doppler window W = 2*half_width+1 with half_width %d exceeds n_dop_c = %d", hw, full);
        return fail(ACQ_ERR_ARG, "Doppler window W = 2*half_width+1 = %d exceeds n_dop = %d", 2 * hw + 1, full);
    }
    if (!packed || !out) return fail(ACQ_ERR_ARG, "packed/out must not be NULL");
    if (n_captures <= 0) return fail(ACQ_ERR_ARG, "n_captures must be > 0 (got %d)", n_captures);
    if ((long long)n_captures * K * e->n_shift > (1 << 24)) return fail(ACQ_ERR_ARG, "too many capture blocks");
    if (e->pending) return fail(ACQ_ERR_ARG, "a submitted search is still pending: call acq_wait first");
    if (device && ((uintptr_t)packed & 15) != 0)
        return fail(ACQ_ERR_ARG, "packed_dev must be 16-byte aligned (the front end stages it with bulk async copies)");
    // A non-coherent search forgets the last search (of either kind) from here on, also when it is refused below; a
    // refused coherent search leaves it.
    if (!m.coherent) e->last = e->last_coh = {};
    if (m.coherent && K % m.m_coh) return fail(ACQ_ERR_ARG, "k_noncoh=%d is not a multiple of m_coh=%d", K, m.m_coh);
    const int n_sats = (int)e->sats.size();
    if (sel && n_sel <= 0) return fail(ACQ_ERR_ARG, "n_sel must be > 0 when sel is given");
    const int n_slots = sel ? n_sel : n_sats;
    for (int i = 0; sel && i < n_sel; i++)
        if (sel[i] < 0 || sel[i] >= n_sats)
            return fail(ACQ_ERR_ARG, "satellite index %d outside the table (0..%d)", sel[i], n_sats - 1);
    if (m.coherent) {
        if (e->prm.code_doppler)
            return fail(ACQ_ERR_UNSUPPORTED, "coherent search of a code_doppler engine is not implemented");
        for (int i = 0; i < n_slots; i++)
            if (e->sats[sel ? sel[i] : i].type == ACQ_E1B)
                return fail(ACQ_ERR_UNSUPPORTED, "coherent search of E1B rows is not implemented (satellite %d): E1B "
                            "symbols drift against the block edges", sel ? sel[i] : i);
        if ((long long)n_captures * K * m.variants(e) > (1 << 24))
            return fail(ACQ_ERR_UNSUPPORTED, "coherent search too large for one call (more than 2^24 capture spectra): split the captures");
    }
    if ((double)n_captures * (double)n_slots * (double)m.dops(e) > (double)acq::kMaxTilesPerLaunch)
        return fail(ACQ_ERR_UNSUPPORTED, "%ssearch too large for one call (more than 2^31 - 1 tiles): split the captures",
                    m.coherent ? "coherent " : "");
    return ACQ_OK;
}

// Enqueue front end + forward FFT + search (which ends in the best-Doppler pick) on `st` for captures already on the
// device, in mode m with m.center on the device.  records_dev: where the kernels write the records (device memory, or the
// device alias of mapped host memory); flag_dev: mapped completion word, or NULL.
int enqueue_search(acq_engine *e, const SearchMode &m, const uint8_t *packed_dev, int n_captures, acq_record *records_dev,
                   unsigned *flag_dev, cudaStream_t st, const uint8_t *packed_host_arg)
{
    const int K = e->prm.k_noncoh;
    const int n_dop = m.dops(e), nvar = m.variants(e);
    const int blocks = n_captures * K;
    const bool prof = e->profiling;
    int rc = wait_scratch(e, st, false);
    if (rc) return rc;
    // Programmatic dependent launch between the kernels of a search: a gain where the search is a few waves of tiles
    // (single captures: 85 -> 77 us for the reference's 32-PRN cold start) and, since every kernel of the chain asks for
    // the same shared-memory carveout (search_kernels_configure), a small one on long searches too (K = 20: 3.453 ->
    // 3.437 ms, E1B with K = 4: 0.709 -> 0.702 ms, a 128-capture farm 5.97 -> 5.95 ms).  Before that it cost long searches
    // 3 %: an SM had to empty before it could change its split, so the search CTAs of the early-launched grid were placed
    // unevenly.  Event records between the kernels (profiling) would serialise them anyway.
    const bool pdl = !prof;
    if (++e->epoch >= 0xfffffffeu) e->epoch = 1;
    if (prof) CU(cudaEventRecord(e->prof[0], st));
    if (packed_host_arg) {   // one 1-bit block still in host memory: it rides in the front end's launch
        if (!launch_front_end_arg(packed_host_arg, e->d_x2, e->d_rot, e->nvar, e->n_shift, e->smax, st))
            return fail(ACQ_ERR_CUDA, "front-end launch failed: %s", cudaGetErrorString(cudaGetLastError()));
        e->launches++;
    } else {
        // a coherent search: k_front_end writes variant 0 (and with F = 2 variant 1, from row 1 of the table, which equals
        // the half-bin table), k_coh_variants the others
        const float2 *rot = m.coherent ? e->d_rot_coh[m.m_coh] + kN : e->d_rot;
        e->launches += launch_front_end(packed_dev, e->d_x2, rot, blocks, nvar, K, e->sample_bits, e->n_shift, e->smax, st);
        if (nvar > 2) e->launches += launch_coh_variants(e->d_x2, e->d_rot_coh[m.m_coh], blocks, nvar, K, st);
    }
    if (prof) CU(cudaEventRecord(e->prof[1], st));
    e->launches += launch_fwd_fft(e->d_x2, e->d_Dp, e->d_tables, blocks * nvar * e->n_shift, true, e->sm_count, st, pdl);
    if (prof) CU(cudaEventRecord(e->prof[2], st));
    SearchArgs a{};
    a.Dp = e->d_Dp;
    a.Ep = e->d_Ep;
    a.tables = e->d_tables;
    a.cells = e->d_cells;
    a.n_slots = e->n_slots;
    a.n_dop = n_dop;
    a.dop_lo = e->prm.dop_lo * m.dop_scale();
    a.dop_center = m.center;
    a.half_width = m.half_width;
    a.dop_hi = e->prm.dop_hi * m.dop_scale();
    a.half_bin = e->prm.half_bin;
    a.K = K;
    a.nvar = nvar;
    a.ext_len = e->ext_len;
    a.Q = e->Q;
    a.n_shift = e->n_shift;
    a.smax = e->smax;
    a.cd_div = e->cd_div;
    const int n_rows = n_captures * e->n_slots;
    const bool fold = n_rows <= kFoldPickRowsMax;
    const long long tiles_l1 = (long long)n_captures * e->n_l1 * n_dop, tiles_e1b = (long long)n_captures * e->n_e1b * n_dop;
    const int kind_l1 = m.coherent ? kSearchL1Coh : search_kind_l1(K, e->prm.half_bin);
    a.ctas_done = e->d_ctas_done;
    a.ctas_total = fold ? (unsigned)(search_grid_ctas(tiles_l1, kind_l1, e->sm_count) +
                                     search_grid_ctas(tiles_e1b, search_kind_e1b(tiles_e1b, e->sm_count), e->sm_count))
                        : 0u;
    a.wait_prior = 1;
    if (e->n_l1 > 0) {   // a coherent search has no E1B row (check_search)
        a.work = e->cur_work;
        a.n_work = e->n_l1;
        a.n_tiles = tiles_l1;
        a.tile_ctr = e->d_tile_ctr;
        e->launches += m.coherent ? launch_search_coh(CohSearchArgs(a, m.m_coh), e->sm_count, st, pdl)
                                  : launch_search(a, false, e->sm_count, st, pdl);
        // The C/A kernel raises its launch-dependents trigger only after its own wait for the forward FFT, so an E1B
        // launch chained to it by programmatic dependent launch starts with the capture spectra complete: it does
        // not wait again, and its CTAs move in as the C/A kernel's last CTAs retire (the two write disjoint rows, and
        // k_pick_small counts finished CTAs of both launches: nothing downstream needs them to finish in order).
        if (pdl && fold) a.wait_prior = 0;
    }
    if (e->n_e1b > 0) {
        a.work = e->cur_work + e->n_l1;
        a.n_work = e->n_e1b;
        a.n_tiles = tiles_e1b;
        a.tile_ctr = e->d_tile_ctr + 1;
        e->launches += launch_search(a, true, e->sm_count, st, pdl);
    }
    if (prof) CU(cudaEventRecord(e->prof[3], st));
    const PickDop pd{a.dop_lo, m.center, m.half_width, a.dop_hi};
    if (fold)
        e->launches += launch_pick_small(e->d_cells, e->cur_slot_sat, records_dev, e->d_ctas_done, a.ctas_total, flag_dev,
                                         e->epoch, n_rows, e->n_slots, n_dop, pd, st, pdl);
    else
        e->launches += launch_best_dop(e->d_cells, e->cur_slot_sat, records_dev, n_captures, e->n_slots, n_dop, pd, st, pdl);
    if (prof) {
        CU(cudaEventRecord(e->prof[4], st));
        e->prof_valid = true;
    }
    CU(cudaGetLastError());
    return ACQ_OK;
}

// Wait for a host-polled search and collect its records: k_pick_small writes every record into mapped memory as two
// 16-byte halves that each end in the search's epoch (acq_record_tagged), so a half whose tag matches has arrived whole.
// The stream is queried now and then so that a failed launch cannot hang the caller; the mapped word *h_flag is only
// ever written to report that the pick gave up (0xffffffff).
int poll_records(acq_engine *e, acq_record *out, size_t rows)
{
    const volatile acq_record_tagged *h = e->h_records.p;
    const unsigned epoch = e->epoch;
    unsigned spins = 0;
    for (size_t i = 0; i < rows; i++) {
        while (h[i].tag0 != epoch || h[i].tag1 != epoch) {
            if ((++spins & 0x3ff) == 0) {
                if (*(volatile unsigned *)e->h_flag.p == 0xffffffffu) {
                    *e->h_flag.p = 0;
                    return fail(ACQ_ERR_CUDA, "search kernels did not complete (best-Doppler pick timed out)");
                }
                const cudaError_t q = cudaStreamQuery(e->stream);
                if (q != cudaSuccess && q != cudaErrorNotReady) return fail(ACQ_ERR_CUDA, "search failed: %s", cudaGetErrorString(q));
                if (q == cudaSuccess && (h[i].tag0 != epoch || h[i].tag1 != epoch))
                    return fail(ACQ_ERR_CUDA, "search finished without delivering its records");
            }
#if defined(__x86_64__) || defined(__i386__)
            __builtin_ia32_pause();  // a polite spin: the wait is tens of microseconds
#endif
        }
        out[i].sat = h[i].sat;
        out[i].lag = h[i].lag;
        out[i].dop = h[i].dop;
        out[i].peak = h[i].peak;
        out[i].noise = h[i].noise;
        out[i].snr = h[i].snr;
    }
    return ACQ_OK;
}

// Host path.  center (HOST, one per row) of an aided mode is staged through pinned memory.
int search_host(acq_engine *e, const SearchMode &m, const uint8_t *packed, int n_captures, const int32_t *sel, int n_sel,
                acq_record *out, acq_cell *grid, bool sync)
{
    int rc = check_search(e, m, packed, n_captures, sel, n_sel, out, false);
    if (rc) return rc;
    DeviceGuard g(e->device);
    e->last = e->last_coh = {};  // until this search is enqueued, there are no spectra refinement or profile could use
    if ((rc = set_selection(e, sel, n_sel)) || (rc = ensure_scratch(e, n_captures, true, m))) return rc;
    const int n_dop = m.dops(e);
    const size_t bytes = (size_t)n_captures * e->prm.k_noncoh * e->block_bytes;
    const size_t rows = (size_t)n_captures * e->n_slots;
    const bool host_records = rows <= (size_t)kHostRecordRowsMax;
    const long long tiles_total = (long long)rows * n_dop * e->prm.k_noncoh;
    const bool poll = host_records && sync && !grid && !e->profiling && tiles_total <= 64LL * e->sm_count;
    // The reference's own search -- one 1-bit block (gps/search.cpp:389-411) -- hands its 8 KiB to the front end as a
    // kernel argument: the launch carries the bytes, nothing is staged or copied ahead of the first kernel.
    const bool as_arg = ACQ_ARG_INPUT && !m.coherent && n_captures == 1 && e->prm.k_noncoh == 1 && e->sample_bits == 1 &&
                        bytes == (size_t)ACQ_BLOCK_BYTES;
    const uint8_t *src = packed;
    if (!as_arg) {
        if (bytes <= kStagePackedMax) {
            memcpy(e->h_packed.p, packed, bytes);
            src = e->h_packed.p;
        }
        CU(cudaMemcpyAsync(e->d_packed, src, bytes, cudaMemcpyHostToDevice, e->stream));
    }
    SearchMode dm = m;
    if (m.aided) {   // from pinned memory: an asynchronous copy node ahead of the front end, even when the capture rides as an argument
        memcpy(e->h_center.p, m.center, rows * sizeof(int32_t));
        CU(cudaMemcpyAsync(e->d_center, e->h_center.p, rows * sizeof(int32_t), cudaMemcpyHostToDevice, e->stream));
        dm.center = e->d_center;
    }
    acq_record *records_dev = host_records ? reinterpret_cast<acq_record *>(e->h_records.dev) : e->d_records.p;
    if ((rc = enqueue_search(e, dm, e->d_packed, n_captures, records_dev, poll ? e->h_flag.dev : nullptr, e->stream,
                             as_arg ? packed : nullptr)))
        return rc;
    if (!m.coherent) e->last = {n_captures, e->n_slots, e->n_l1, e->n_e1b, e->cur_slot_sat, true};
    else e->last_coh = {n_captures, e->n_slots, e->n_l1, e->n_e1b, e->cur_slot_sat, true, m.m_coh};
    if (!host_records) CU(cudaMemcpyAsync(out, e->d_records, rows * sizeof(acq_record), cudaMemcpyDeviceToHost, e->stream));
    if (grid)
        CU(cudaMemcpyAsync(grid, e->d_cells, rows * n_dop * sizeof(acq_cell), cudaMemcpyDeviceToHost, e->stream));
    if (!sync) {
        CU(cudaEventRecord(e->done, e->stream));
        e->pending = true;
        e->pending_rows = host_records ? (int)rows : 0;
        e->pending_out = out;
        return ACQ_OK;
    }
    if (poll) {
        if ((rc = poll_records(e, out, rows))) return rc;
    } else {
        CU(cudaStreamSynchronize(e->stream));
        if (host_records) memcpy(out, e->h_records.p, rows * sizeof(acq_record));
    }
    e->dev_pending = false;  // this search was ordered behind the last device-path work, so that is complete too
    return ACQ_OK;
}

// completion of an acq_submit: records that the kernels left in the mapped buffer go to the caller's array
void finish_pending(acq_engine *e)
{
    if (e->pending_rows > 0 && e->pending_out)
        memcpy(e->pending_out, e->h_records.p, (size_t)e->pending_rows * sizeof(acq_record));
    e->pending = false;
    e->pending_rows = 0;
    e->pending_out = nullptr;
}

// Device path: packed_dev, out_dev and the centres of an aided mode are the caller's device arrays
int search_device(acq_engine *e, const SearchMode &m, const uint8_t *packed_dev, int n_captures, const int32_t *sel,
                  int n_sel, acq_record *out_dev, void *stream)
{
    int rc = check_search(e, m, packed_dev, n_captures, sel, n_sel, out_dev, true);
    if (rc) return rc;
    DeviceGuard g(e->device);
    e->last = e->last_coh = {};  // refinement and profile apply once this search is enqueued
    if ((rc = set_selection(e, sel, n_sel)) || (rc = ensure_scratch(e, n_captures, false, m))) return rc;
    cudaStream_t st = stream ? (cudaStream_t)stream : e->stream;
    if ((rc = enqueue_search(e, m, packed_dev, n_captures, out_dev, nullptr, st, nullptr))) return rc;
    if (!m.coherent) e->last = {n_captures, e->n_slots, e->n_l1, e->n_e1b, e->cur_slot_sat, false};
    else e->last_coh = {n_captures, e->n_slots, e->n_l1, e->n_e1b, e->cur_slot_sat, false, m.m_coh};
    return hold_scratch(e, st);
}

// The search acq_refine* and acq_profile* apply to (last), or acq_refine_coherent* and acq_profile_coherent* (last_coh)
const acq_engine::LastSearch &last_of(const acq_engine *e, bool coherent) { return coherent ? e->last_coh : e->last; }

// The checks of acq_refine* and acq_profile* (`what`) against the last search, after those of their own arguments.
// The host forms take the records of a host-path search and check each one here; the device forms leave that to the
// kernels, which write a marker row for a record that fails.  coherent: the checks of the coherent forms, against the
// last coherent search, whose records' Doppler indices run over M dop_lo .. M dop_hi.
int check_records(acq_engine *e, const acq_record *rec, int n_records, bool device, bool coherent, const char *what)
{
    if (e->pending) return fail(ACQ_ERR_ARG, "a submitted search is still pending: call acq_wait first");
    const acq_engine::LastSearch &ls = last_of(e, coherent);
    const char *kind = coherent ? "coherent " : "";
    if (device && ls.captures <= 0)
        return fail(ACQ_ERR_ARG, "no %ssearch whose spectra are still on the device to %s", kind, what);
    if (!device && (ls.captures <= 0 || !ls.host))
        return fail(ACQ_ERR_ARG, "no completed host-path %ssearch to %s", kind, what);
    const long long rows = (long long)ls.captures * ls.slots;
    if (n_records != rows)
        return fail(ACQ_ERR_ARG, "n_records=%d but the last %ssearch produced %lld records", n_records, kind, rows);
    if (device) return ACQ_OK;
    const int M = coherent ? ls.m_coh : 1, lo = M * e->prm.dop_lo, hi = M * e->prm.dop_hi;
    for (int i = 0; i < n_records; i++) {
        const acq_record &r = rec[i];
        if (r.sat != e->sel_cache[i % ls.slots])
            return fail(ACQ_ERR_ARG, "record %d: sat %d is not the satellite searched in that slot", i, r.sat);
        const int L = (e->sats[r.sat].type == ACQ_E1B) ? ACQ_LAGS_E1B : ACQ_LAGS_L1;
        if (r.lag < 0 || r.lag >= L) return fail(ACQ_ERR_ARG, "record %d: lag %d outside 0..%d", i, r.lag, L - 1);
        // a row that never exceeded snr 0 carries dop 0 (k_best_dop), which may lie outside an asymmetric range
        if ((r.dop < lo || r.dop > hi) && !(r.dop == 0 && r.snr == 0.0f))
            return fail(ACQ_ERR_ARG, "record %d: Doppler index %d outside %d..%d", i, r.dop, lo, hi);
    }
    return ACQ_OK;
}

// excl of acq_profile against the search it follows: 0 <= excl < L_min / 2, L_min the smallest L of its satellites
int check_excl(int excl, int n_l1)
{
    const int l_min = n_l1 > 0 ? ACQ_LAGS_L1 : ACQ_LAGS_E1B;
    if (excl < 0 || 2 * excl >= l_min)
        return fail(ACQ_ERR_ARG, "excl=%d outside 0..%d (L_min / 2 - 1 of the searched satellites)", excl, (l_min - 1) / 2);
    return ACQ_OK;
}

// Lag-vector floats of one capture's rows (acq_b200.h: L per slot)
size_t profile_capture_len(int n_l1, int n_e1b) { return (size_t)n_l1 * ACQ_LAGS_L1 + (size_t)n_e1b * ACQ_LAGS_E1B; }

// The arguments refinement and profile share: the spectra and shape of the last search (A::kCoh: the last coherent search,
// its F variants per block and its M times finer Doppler range), the records and the flags.  A coherent form's min_snr is
// the threshold of its DETECTED flag (set when min_snr > 0).
template <class A>
A last_search_args(const acq_engine *e, const acq_record *rec_dev, int flags, float min_snr)
{
    constexpr bool coherent = A::kCoh;
    const acq_engine::LastSearch &ls = last_of(e, coherent);
    const int M = coherent ? ls.m_coh : 1;
    A a{};
    a.Dp = e->d_Dp;
    a.Ep = e->d_Ep;
    a.rec = rec_dev;
    a.sat_type = e->d_sat_type;
    a.slot_sat = ls.slot_sat;
    a.n_slots = ls.slots;
    a.K = e->prm.k_noncoh;
    a.nvar = coherent ? M * (1 + e->prm.half_bin) : e->nvar;
    a.half_bin = e->prm.half_bin;
    a.ext_len = e->ext_len;
    a.Q = e->Q;
    a.n_shift = e->n_shift;
    a.smax = e->smax;
    a.cd_div = e->cd_div;
    a.n_sats = (int)e->sats.size();
    a.dop_lo = M * e->prm.dop_lo;
    a.dop_hi = M * e->prm.dop_hi;
    a.flags = flags;
    a.thr_l1 = coherent ? min_snr : e->prm.thr_l1;
    a.thr_e1b = coherent ? min_snr : e->prm.thr_e1b;
    if constexpr (coherent) a.m_coh = M;
    return a;
}

int enqueue_refine(acq_engine *e, bool coherent, const acq_record *rec_dev, int n_records, int flags, float min_snr,
                   acq_fine *out_dev, cudaStream_t st)
{
    auto launch = [&](auto a) {
        a.out = out_dev;
        return launch_refine(a, n_records, st);
    };
    e->launches += coherent ? launch(last_search_args<RefineCohArgs>(e, rec_dev, flags, min_snr))
                            : launch(last_search_args<RefineArgs>(e, rec_dev, flags, min_snr));
    CU(cudaGetLastError());
    return ACQ_OK;
}

int enqueue_profile(acq_engine *e, bool coherent, const acq_record *rec_dev, int n_records, int flags, float min_snr,
                    int excl, acq_peak2 *out_dev, float *profile_dev, cudaStream_t st)
{
    auto launch = [&](auto a) {
        a.tables = e->d_tables;
        a.out = out_dev;
        a.profile = profile_dev;
        a.n_e1b_slots = last_of(e, coherent).n_e1b;   // 0 after a coherent search (C/A rows only, check_search)
        a.excl = excl;
        return launch_profile(a, n_records, st);
    };
    e->launches += coherent ? launch(last_search_args<ProfileCohArgs>(e, rec_dev, flags, min_snr))
                            : launch(last_search_args<ProfileArgs>(e, rec_dev, flags, min_snr));
    CU(cudaGetLastError());
    return ACQ_OK;
}

// acq_refine / acq_refine_coherent after their argument checks: the records go to the device, are refined on the engine
// stream and come back.  The records are checked here, so the kernel's own checks pass every row.
int refine_host(acq_engine *e, bool coherent, const acq_record *rec, int n_records, acq_fine *out)
{
    int rc = check_records(e, rec, n_records, false, coherent, "refine");
    if (rc) return rc;
    DeviceGuard g(e->device);
    if ((rc = grow(e, e->d_ref_rec, (size_t)n_records)) || (rc = grow(e, e->d_fine, (size_t)n_records))) return rc;
    CU(cudaMemcpyAsync(e->d_ref_rec, rec, (size_t)n_records * sizeof(acq_record), cudaMemcpyHostToDevice, e->stream));
    if ((rc = enqueue_refine(e, coherent, e->d_ref_rec, n_records, 0, 0.0f, e->d_fine, e->stream))) return rc;
    CU(cudaMemcpyAsync(out, e->d_fine, (size_t)n_records * sizeof(acq_fine), cudaMemcpyDeviceToHost, e->stream));
    CU(cudaStreamSynchronize(e->stream));
    return ACQ_OK;
}

// acq_refine_device / acq_refine_coherent_device after their argument checks
int refine_device(acq_engine *e, bool coherent, const acq_record *rec_dev, int n_records, int flags, float min_snr,
                  acq_fine *out_dev, void *stream)
{
    int rc = check_records(e, rec_dev, n_records, true, coherent, "refine");
    if (rc) return rc;
    if (((uintptr_t)out_dev & 15) != 0) return fail(ACQ_ERR_ARG, "out_dev must be 16-byte aligned (one 16-byte store per row)");
    if (((uintptr_t)rec_dev & 3) != 0) return fail(ACQ_ERR_ARG, "rec_dev must be 4-byte aligned");
    DeviceGuard g(e->device);
    cudaStream_t st = stream ? (cudaStream_t)stream : e->stream;
    // after the search that left the spectra (on any stream), before the next search overwrites them
    if ((rc = wait_scratch(e, st, true)) || (rc = enqueue_refine(e, coherent, rec_dev, n_records, flags, min_snr, out_dev, st)))
        return rc;
    return hold_scratch(e, st);
}

// acq_profile / acq_profile_coherent after their argument checks (excl >= 0)
int profile_host(acq_engine *e, bool coherent, const acq_record *rec, int n_records, int excl, acq_peak2 *out, float *profile)
{
    int rc = check_records(e, rec, n_records, false, coherent, "profile");
    const acq_engine::LastSearch &ls = last_of(e, coherent);
    if (rc || (rc = check_excl(excl, ls.n_l1))) return rc;
    DeviceGuard g(e->device);
    const size_t n_prof = (size_t)ls.captures * profile_capture_len(ls.n_l1, ls.n_e1b);
    if ((rc = grow(e, e->d_ref_rec, (size_t)n_records)) || (rc = grow(e, e->d_peak2, (size_t)n_records))) return rc;
    // The lag profiles (512 MiB for a 1024-capture C/A search) live only for this call: the engine keeps no buffer of
    // that size.  The buffer is freed after the engine stream has passed every use of it, on the error paths too.
    struct CallBuffer {
        cudaStream_t st;
        float *p = nullptr;
        ~CallBuffer()
        {
            if (p) {
                cudaStreamSynchronize(st);
                cudaFree(p);
            }
        }
    } d_prof{e->stream};
    if (profile) CU(cudaMalloc(&d_prof.p, n_prof * sizeof(float)));
    CU(cudaMemcpyAsync(e->d_ref_rec, rec, (size_t)n_records * sizeof(acq_record), cudaMemcpyHostToDevice, e->stream));
    // the records are checked above, so the kernel's own checks pass every row
    if ((rc = enqueue_profile(e, coherent, e->d_ref_rec, n_records, 0, 0.0f, excl, e->d_peak2, d_prof.p, e->stream))) return rc;
    CU(cudaMemcpyAsync(out, e->d_peak2, (size_t)n_records * sizeof(acq_peak2), cudaMemcpyDeviceToHost, e->stream));
    if (profile) CU(cudaMemcpyAsync(profile, d_prof.p, n_prof * sizeof(float), cudaMemcpyDeviceToHost, e->stream));
    CU(cudaStreamSynchronize(e->stream));
    return ACQ_OK;
}

// acq_profile_device / acq_profile_coherent_device after their argument checks (excl >= 0)
int profile_device(acq_engine *e, bool coherent, const acq_record *rec_dev, int n_records, int flags, float min_snr, int excl,
                   acq_peak2 *out_dev, float *profile_dev, void *stream)
{
    int rc = check_records(e, rec_dev, n_records, true, coherent, "profile");
    if (rc || (rc = check_excl(excl, last_of(e, coherent).n_l1))) return rc;
    if (((uintptr_t)out_dev & 15) != 0) return fail(ACQ_ERR_ARG, "out_dev must be 16-byte aligned (one 16-byte store per row)");
    if (((uintptr_t)rec_dev & 3) != 0) return fail(ACQ_ERR_ARG, "rec_dev must be 4-byte aligned");
    if (((uintptr_t)profile_dev & 3) != 0) return fail(ACQ_ERR_ARG, "profile_dev must be 4-byte aligned");
    DeviceGuard g(e->device);
    cudaStream_t st = stream ? (cudaStream_t)stream : e->stream;
    // ordered as acq_refine_device: after the search that left the spectra, before the next one
    if ((rc = wait_scratch(e, st, true)) ||
        (rc = enqueue_profile(e, coherent, rec_dev, n_records, flags, min_snr, excl, out_dev, profile_dev, st)))
        return rc;
    return hold_scratch(e, st);
}

// min_snr of the coherent device forms: a NaN would skip every row without saying so
int check_min_snr(float min_snr)
{
    if (std::isnan(min_snr)) return fail(ACQ_ERR_ARG, "min_snr is NaN");
    return ACQ_OK;
}

}  // namespace

extern "C" {

const char *acq_last_error(void) { return g_err.c_str(); }
int acq_abi_version(void) { return ACQ_ABI_VERSION; }

int acq_params_default(acq_params *p)
{
    if (!p) return fail(ACQ_ERR_ARG, "params is NULL");
    memset(p, 0, sizeof *p);
    p->struct_size = (uint32_t)sizeof(acq_params);
    p->dop_lo = -20;  // int(-5000/BIN_SIZE), gps/search.cpp:465
    p->dop_hi = 20;
    p->half_bin = 0;
    p->k_noncoh = 1;
    p->thr_l1 = 16.0f;   // MIN_SIG, gps/gps.h:60
    p->thr_e1b = 16.0f;  // gps/search.cpp:549
    p->wrap_mode = ACQ_WRAP_REFERENCE;
    p->sample_bits = 1;  // the sampler's I_sign stream, gps/search.cpp:408-411
    p->code_doppler = 0;
    return ACQ_OK;
}

int acq_create(acq_engine **out, const acq_params *params, const acq_sat *sats, int n_sats, int device)
{
    if (!out) return fail(ACQ_ERR_ARG, "out is NULL");
    *out = nullptr;
    if (!sats || n_sats <= 0 || n_sats > 4096) return fail(ACQ_ERR_ARG, "bad satellite table (n_sats=%d)", n_sats);
    acq_params prm;
    if (params) {
        // the first member is the size of the caller's structure: anything but this library's layout is refused
        // before a byte beyond it is read
        if (params->struct_size != (uint32_t)sizeof(acq_params))
            return fail(ACQ_ERR_ARG, "acq_params.struct_size is %u, this library (ABI version %d) expects %zu: fill the "
                        "structure with acq_params_default() from the matching acq_b200.h", params->struct_size,
                        ACQ_ABI_VERSION, sizeof(acq_params));
        prm = *params;
    } else {
        acq_params_default(&prm);
    }
    if (prm.dop_hi < prm.dop_lo) return fail(ACQ_ERR_ARG, "dop_hi < dop_lo");
    if (prm.k_noncoh < 1 || prm.k_noncoh > 255) return fail(ACQ_ERR_ARG, "k_noncoh must be in 1..255");
    if (prm.half_bin != 0 && prm.half_bin != 1) return fail(ACQ_ERR_ARG, "half_bin must be 0 or 1");
    if (prm.wrap_mode != ACQ_WRAP_REFERENCE && prm.wrap_mode != ACQ_WRAP_CIRCULAR)
        return fail(ACQ_ERR_ARG, "bad wrap_mode");
    if (prm.sample_bits < 0 || prm.sample_bits > 2) return fail(ACQ_ERR_ARG, "sample_bits must be 1 or 2 (0 = 1)");
    if (prm.sample_bits == 0) prm.sample_bits = 1;  // the member used to be "reserved, must be 0"
    if (prm.code_doppler != 0 && prm.code_doppler != 1) return fail(ACQ_ERR_ARG, "code_doppler must be 0 or 1");
    for (int32_t r : prm.reserved)
        if (r) return fail(ACQ_ERR_ARG, "reserved members must be 0");
    // code-Doppler compensation: largest lag shift over the Doppler range, reached in the last block
    const int cd_div = 385 * (prm.half_bin ? 2 : 1);  // FS/DECIM/f_L1 = 4.092e6/1575.42e6 = 1/385 exactly
    int smax = 0;
    if (prm.code_doppler && prm.k_noncoh > 1)
        smax = std::max(std::abs(acq::code_shift(prm.k_noncoh - 1, prm.dop_lo, cd_div)),
                        std::abs(acq::code_shift(prm.k_noncoh - 1, prm.dop_hi, cd_div)));
    if (2 * smax + 1 > ACQ_MAX_CODE_SHIFTS)
        return fail(ACQ_ERR_UNSUPPORTED, "code_doppler needs %d shifted copies of every capture spectrum (limit %d): "
                    "reduce k_noncoh or the Doppler span", 2 * smax + 1, ACQ_MAX_CODE_SHIFTS);
    const int max_idx = std::max(std::abs(prm.dop_lo), std::abs(prm.dop_hi));
    const int max_bins = prm.half_bin ? (max_idx + 1) / 2 + 1 : max_idx;
    if (max_bins > 2048) return fail(ACQ_ERR_ARG, "Doppler span too large (|bins| <= 2048)");
    for (int i = 0; i < n_sats; i++) {
        const acq_sat &s = sats[i];
        if (s.type == ACQ_E1B) {
            if (s.prn < 1 || s.prn > 50) return fail(ACQ_ERR_ARG, "sat %d: E1B prn %d outside 1..50", i, s.prn);
        } else if (s.type == ACQ_NAVSTAR || s.type == ACQ_QZSS || s.type == ACQ_SBAS) {
            const bool preset = (s.t1 > 10 || s.t2 > 10);
            if (!preset && (s.t1 < 1 || s.t2 < 1)) return fail(ACQ_ERR_ARG, "sat %d: G2 taps must be in 1..10", i);
            if (preset && (s.t2 < 0 || s.t2 > 1023)) return fail(ACQ_ERR_ARG, "sat %d: G2 preset out of range", i);
        } else {
            return fail(ACQ_ERR_ARG, "sat %d: unknown type %d", i, s.type);
        }
    }

    int n_dev = 0;
    if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev == 0) {
        cudaGetLastError();
        return fail(ACQ_ERR_NO_DEVICE, "no CUDA device available (this engine has no CPU fallback)");
    }
    if (device < 0 || device >= n_dev) return fail(ACQ_ERR_ARG, "device %d out of range (0..%d)", device, n_dev - 1);
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10)
        return fail(ACQ_ERR_NO_DEVICE, "device %d is sm_%d%d; this library is built for sm_100a only", device,
                    prop.major, prop.minor);

    DeviceGuard g(device);
    std::unique_ptr<acq_engine> e(new acq_engine);   // freed on every error return below
    e->device = device;
    e->sm_count = prop.multiProcessorCount;
    e->sm_clock_khz = prop.clockRate;
    e->prm = prm;
    e->sats.assign(sats, sats + n_sats);
    e->n_dop = prm.dop_hi - prm.dop_lo + 1;
    e->nvar = prm.half_bin ? 2 : 1;
    e->smax = smax;
    e->n_shift = 2 * smax + 1;
    e->cd_div = cd_div;
    e->sample_bits = prm.sample_bits;
    e->block_bytes = ACQ_CAPTURE_BLOCK_BYTES(prm.sample_bits);
    e->Q = max_bins / 4 + 2;
    e->ext_len = kSub + 2 * e->Q;

    CU(cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking));
    CU(cudaEventCreateWithFlags(&e->done, cudaEventDisableTiming));
    CU(cudaEventCreateWithFlags(&e->dev_done, cudaEventDisableTiming));
    CU(search_kernels_configure());
    // completion counter of small searches, mapped completion word
    CU(e->d_ctas_done.alloc(1));
    CU(cudaMemset(e->d_ctas_done, 0, sizeof(unsigned)));
    CU(e->d_tile_ctr.alloc(4));
    CU(cudaMemset(e->d_tile_ctr, 0, 4 * sizeof(unsigned)));
    CU(e->h_flag.alloc(1));
    {   // work lists that need no upload: the whole table (C/A rows first, then E1B) and every single satellite
        std::vector<int2> full, single(n_sats);
        std::vector<int> ident(n_sats);
        for (int pass = 0; pass < 2; pass++)
            for (int i = 0; i < n_sats; i++) {
                const bool e1b = (sats[i].type == ACQ_E1B);
                if ((pass == 1) != e1b) continue;
                full.push_back(make_int2(i, i));
                if (!e1b) e->full_n_l1++;
            }
        for (int i = 0; i < n_sats; i++) {
            single[i] = make_int2(i, 0);
            ident[i] = i;
        }
        CU(upload(e->d_work_full, full));
        CU(upload(e->d_work_single, single));
        CU(upload(e->d_sat_full, ident));
    }

    // ---- twiddle tables, constants (double precision on the host, rounded once)
    const double two_pi = 6.283185307179586476925286766559;
    std::vector<float2> tables(kT2Elems + kBaseElems);
    for (int k2 = 0; k2 < 4; k2++)
        for (int n1 = 1; n1 < 16; n1++)
            for (int c = 0; c < 16; c++) {
                const double a = two_pi * (double)(((4 * c + k2) * n1) % 1024) / 1024.0;
                tables[(k2 * 15 + (n1 - 1)) * 16 + c] = make_float2((float)cos(a), (float)sin(a));
            }
    for (int k2 = 0; k2 < 4; k2++)
        for (int t = 0; t < 256; t++) {
            const double a = two_pi * (double)(4 * t + k2) / 16384.0;
            tables[kT2Elems + k2 * 256 + t] = make_float2((float)cos(a), (float)sin(a));
        }
    float2 cC[64];
    for (int k2 = 0; k2 < 4; k2++)
        for (int n = 0; n < 16; n++) {
            const double c = two_pi * (double)(k2 * n) / 64.0;
            cC[k2 * 16 + n] = make_float2((float)cos(c), (float)sin(c));
        }
    // Half-band taps of the reference (gps/search.cpp:101-136, column 0), narrowed double -> float the
    // way its initialiser does, in application order: COEF[0], COEF[2..30 step 2], COEF[15].
    static const double taps_even[16] = {-0.010233, 0.010668, -0.016324, 0.024377, -0.036482, 0.056990,
                                         -0.101993, 0.316926, 0.316926,  -0.101993, 0.056990, -0.036482,
                                         0.024377,  -0.016324, 0.010668, -0.010233};
    float hb[17];
    for (int i = 0; i < 16; i++) hb[i] = (float)taps_even[i];
    hb[16] = (float)0.500009;
    CU(launch_tables_init(cC, hb));
    CU(upload(e->d_tables, tables));
    {
        std::vector<int> types(n_sats);
        for (int i = 0; i < n_sats; i++) types[i] = sats[i].type;
        CU(upload(e->d_sat_type, types));
    }
    if (e->nvar == 2) CU(upload(e->d_rot, rotation_table(2, 1)));   // the half-bin rotation exp(-i pi n / N)

    // ---- code spectra (replaces the loops at gps/search.cpp:243-346)
    std::vector<uint32_t> chips((size_t)n_sats * 128);
    std::vector<int> codelen_boc((size_t)n_sats * 2);
    for (int i = 0; i < n_sats; i++) {
        if (sats[i].type == ACQ_E1B) {
            memcpy(&chips[(size_t)i * 128], &kE1bWords[(sats[i].prn - 1) * 128], 128 * sizeof(uint32_t));
            codelen_boc[2 * i] = 4092;
            codelen_boc[2 * i + 1] = 1;
        } else {
            ca_code_bits(sats[i].t1, sats[i].t2, &chips[(size_t)i * 128]);
            // SearchInit builds replicas for Navstar and QZSS rows only (gps/search.cpp:244): an SBAS row of the
            // table keeps the all-zero spectrum of the reference's static code[] array (codelen 0 = no replica)
            codelen_boc[2 * i] = (sats[i].type == ACQ_SBAS) ? 0 : 1023;
            codelen_boc[2 * i + 1] = 0;
        }
    }
    DevBuf<uint32_t> d_chips;
    DevBuf<int> d_clb;
    DevBuf<float2> d_x1, d_x2;
    CU(upload(d_chips, chips));
    CU(upload(d_clb, codelen_boc));
    CU(d_x1.alloc((size_t)n_sats * 32768));
    CU(d_x2.alloc((size_t)n_sats * kN));
    CU(e->d_C.alloc((size_t)n_sats * kN));
    CU(e->d_Ep.alloc((size_t)n_sats * 4 * e->ext_len));
    e->launches += launch_hb1_code(d_chips, d_clb, d_x1, n_sats, e->stream);
    e->launches += launch_hb2(d_x1, d_x2, nullptr, n_sats, 1, 1, e->stream);
    e->launches += launch_fwd_fft(d_x2, e->d_C, e->d_tables, n_sats, false, e->sm_count, e->stream);
    e->launches += launch_build_ext(e->d_C, e->d_Ep, n_sats, e->Q, e->ext_len, prm.wrap_mode, e->stream);
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(e->stream));
    *out = e.release();
    return ACQ_OK;
}

int acq_destroy(acq_engine *e)
{
    if (e) {
        DeviceGuard g(e->device);   // the engine's memory is freed under its own device
        delete e;
    }
    return ACQ_OK;
}

int acq_search(acq_engine *e, const uint8_t *packed, int n_captures, const int32_t *sel, int n_sel, acq_record *out)
{
    return search_host(e, kFullRange, packed, n_captures, sel, n_sel, out, nullptr, true);
}

int acq_search_grid(acq_engine *e, const uint8_t *packed, int n_captures, const int32_t *sel, int n_sel,
                    acq_record *out, acq_cell *grid)
{
    if (!grid) return fail(ACQ_ERR_ARG, "grid is NULL");
    return search_host(e, kFullRange, packed, n_captures, sel, n_sel, out, grid, true);
}

int acq_search_aided(acq_engine *e, const uint8_t *packed, int n_captures, const int32_t *sel, int n_sel,
                     const int32_t *dop_center, int half_width, acq_record *out, acq_cell *grid)
{
    return search_host(e, {true, false, dop_center, half_width, 0}, packed, n_captures, sel, n_sel, out, grid, true);
}

int acq_search_device(acq_engine *e, const uint8_t *packed_dev, int n_captures, const int32_t *sel, int n_sel,
                      acq_record *out_dev, void *stream)
{
    return search_device(e, kFullRange, packed_dev, n_captures, sel, n_sel, out_dev, stream);
}

int acq_search_aided_device(acq_engine *e, const uint8_t *packed_dev, int n_captures, const int32_t *sel, int n_sel,
                            const int32_t *dop_center_dev, int half_width, acq_record *out_dev, void *stream)
{
    return search_device(e, {true, false, dop_center_dev, half_width, 0}, packed_dev, n_captures, sel, n_sel, out_dev, stream);
}

int acq_search_coherent(acq_engine *e, const uint8_t *packed, int n_captures, const int32_t *sel, int n_sel, int m_coh,
                        acq_record *out, acq_cell *grid)
{
    return search_host(e, {false, true, nullptr, 0, m_coh}, packed, n_captures, sel, n_sel, out, grid, true);
}

int acq_search_coherent_device(acq_engine *e, const uint8_t *packed_dev, int n_captures, const int32_t *sel, int n_sel,
                               int m_coh, acq_record *out_dev, void *stream)
{
    return search_device(e, {false, true, nullptr, 0, m_coh}, packed_dev, n_captures, sel, n_sel, out_dev, stream);
}

int acq_search_coherent_aided(acq_engine *e, const uint8_t *packed, int n_captures, const int32_t *sel, int n_sel,
                              int m_coh, const int32_t *dop_center, int half_width, acq_record *out, acq_cell *grid)
{
    return search_host(e, {true, true, dop_center, half_width, m_coh}, packed, n_captures, sel, n_sel, out, grid, true);
}

int acq_search_coherent_aided_device(acq_engine *e, const uint8_t *packed_dev, int n_captures, const int32_t *sel,
                                     int n_sel, int m_coh, const int32_t *dop_center_dev, int half_width,
                                     acq_record *out_dev, void *stream)
{
    return search_device(e, {true, true, dop_center_dev, half_width, m_coh}, packed_dev, n_captures, sel, n_sel, out_dev,
                         stream);
}

int acq_submit(acq_engine *e, const uint8_t *packed, int n_captures, const int32_t *sel, int n_sel, acq_record *out)
{
    return search_host(e, kFullRange, packed, n_captures, sel, n_sel, out, nullptr, false);
}

int acq_poll(acq_engine *e)
{
    if (!e) return fail(ACQ_ERR_ARG, "engine is NULL");
    if (!e->pending) return 1;
    DeviceGuard g(e->device);
    cudaError_t q = cudaEventQuery(e->done);
    if (q == cudaSuccess) {
        finish_pending(e);
        return 1;
    }
    if (q == cudaErrorNotReady) return 0;
    e->pending = false;
    return fail(ACQ_ERR_CUDA, "cudaEventQuery: %s", cudaGetErrorString(q));
}

int acq_wait(acq_engine *e)
{
    if (!e) return fail(ACQ_ERR_ARG, "engine is NULL");
    if (!e->pending) return ACQ_OK;
    DeviceGuard g(e->device);
    const cudaError_t w = cudaEventSynchronize(e->done);
    if (w != cudaSuccess) {
        e->pending = false;
        return fail(ACQ_ERR_CUDA, "cudaEventSynchronize: %s", cudaGetErrorString(w));
    }
    finish_pending(e);
    return ACQ_OK;
}

int acq_refine(acq_engine *e, const acq_record *rec, int n_records, acq_fine *out)
{
    if (!e) return fail(ACQ_ERR_ARG, "engine is NULL");
    if (!rec || !out) return fail(ACQ_ERR_ARG, "rec/out must not be NULL");
    return refine_host(e, false, rec, n_records, out);
}

int acq_refine_device(acq_engine *e, const acq_record *rec_dev, int n_records, int flags, acq_fine *out_dev, void *stream)
{
    if (!e) return fail(ACQ_ERR_ARG, "engine is NULL");
    if (!rec_dev || !out_dev) return fail(ACQ_ERR_ARG, "rec_dev/out_dev must not be NULL");
    if (flags & ~ACQ_REFINE_DETECTED) return fail(ACQ_ERR_ARG, "unknown flag bits 0x%x", (unsigned)(flags & ~ACQ_REFINE_DETECTED));
    return refine_device(e, false, rec_dev, n_records, flags, 0.0f, out_dev, stream);
}

int acq_refine_coherent(acq_engine *e, const acq_record *rec, int n_records, acq_fine *out)
{
    if (!e) return fail(ACQ_ERR_ARG, "engine is NULL");
    if (!rec || !out) return fail(ACQ_ERR_ARG, "rec/out must not be NULL");
    return refine_host(e, true, rec, n_records, out);
}

int acq_refine_coherent_device(acq_engine *e, const acq_record *rec_dev, int n_records, float min_snr, acq_fine *out_dev,
                               void *stream)
{
    if (!e) return fail(ACQ_ERR_ARG, "engine is NULL");
    if (!rec_dev || !out_dev) return fail(ACQ_ERR_ARG, "rec_dev/out_dev must not be NULL");
    int rc = check_min_snr(min_snr);
    if (rc) return rc;
    return refine_device(e, true, rec_dev, n_records, min_snr > 0.0f ? ACQ_REFINE_DETECTED : 0, min_snr, out_dev, stream);
}

int acq_profile(acq_engine *e, const acq_record *rec, int n_records, int excl, acq_peak2 *out, float *profile)
{
    if (!e) return fail(ACQ_ERR_ARG, "engine is NULL");
    if (!rec || !out) return fail(ACQ_ERR_ARG, "rec/out must not be NULL");
    if (excl < 0) return fail(ACQ_ERR_ARG, "excl must be >= 0 (got %d)", excl);
    return profile_host(e, false, rec, n_records, excl, out, profile);
}

int acq_profile_device(acq_engine *e, const acq_record *rec_dev, int n_records, int flags, int excl, acq_peak2 *out_dev,
                       float *profile_dev, void *stream)
{
    if (!e) return fail(ACQ_ERR_ARG, "engine is NULL");
    if (!rec_dev || !out_dev) return fail(ACQ_ERR_ARG, "rec_dev/out_dev must not be NULL");
    if (flags & ~ACQ_PROFILE_DETECTED) return fail(ACQ_ERR_ARG, "unknown flag bits 0x%x", (unsigned)(flags & ~ACQ_PROFILE_DETECTED));
    if (excl < 0) return fail(ACQ_ERR_ARG, "excl must be >= 0 (got %d)", excl);
    return profile_device(e, false, rec_dev, n_records, flags, 0.0f, excl, out_dev, profile_dev, stream);
}

int acq_profile_coherent(acq_engine *e, const acq_record *rec, int n_records, int excl, acq_peak2 *out, float *profile)
{
    if (!e) return fail(ACQ_ERR_ARG, "engine is NULL");
    if (!rec || !out) return fail(ACQ_ERR_ARG, "rec/out must not be NULL");
    if (excl < 0) return fail(ACQ_ERR_ARG, "excl must be >= 0 (got %d)", excl);
    return profile_host(e, true, rec, n_records, excl, out, profile);
}

int acq_profile_coherent_device(acq_engine *e, const acq_record *rec_dev, int n_records, float min_snr, int excl,
                                acq_peak2 *out_dev, float *profile_dev, void *stream)
{
    if (!e) return fail(ACQ_ERR_ARG, "engine is NULL");
    if (!rec_dev || !out_dev) return fail(ACQ_ERR_ARG, "rec_dev/out_dev must not be NULL");
    int rc = check_min_snr(min_snr);
    if (rc) return rc;
    if (excl < 0) return fail(ACQ_ERR_ARG, "excl must be >= 0 (got %d)", excl);
    return profile_device(e, true, rec_dev, n_records, min_snr > 0.0f ? ACQ_PROFILE_DETECTED : 0, min_snr, excl, out_dev,
                          profile_dev, stream);
}

int acq_detected(const acq_engine *e, const acq_record *r)
{
    if (!e || !r || r->sat < 0 || r->sat >= (int)e->sats.size()) return 0;
    const float thr = (e->sats[r->sat].type == ACQ_E1B) ? e->prm.thr_e1b : e->prm.thr_l1;
    return r->snr >= thr ? 1 : 0;  // search.cpp:591: if (snr < min_sig) continue;
}

int acq_get_code_spectrum(acq_engine *e, int sat, float *out)
{
    if (!e || !out) return fail(ACQ_ERR_ARG, "NULL argument");
    if (sat < 0 || sat >= (int)e->sats.size()) return fail(ACQ_ERR_ARG, "sat %d outside the table", sat);
    DeviceGuard g(e->device);
    CU(cudaMemcpy(out, e->d_C + (size_t)sat * kN, kN * sizeof(float2), cudaMemcpyDeviceToHost));
    return ACQ_OK;
}

int acq_get_capture_spectrum(acq_engine *e, const uint8_t *packed, int half_rot, float *x2, float *D)
{
    if (!e || !packed) return fail(ACQ_ERR_ARG, "NULL argument");
    if (half_rot != 0 && half_rot != 1) return fail(ACQ_ERR_ARG, "half_rot must be 0 or 1");
    if (e->pending) return fail(ACQ_ERR_ARG, "a submitted search is still pending");
    DeviceGuard g(e->device);
    DevBuf<uint8_t> d_pk;
    DevBuf<float2> d_x2, d_D, d_rot;
    CU(d_pk.alloc(e->block_bytes));
    CU(d_x2.alloc(2 * kN));
    CU(d_D.alloc(kN));
    CU(cudaMemcpy(d_pk, packed, e->block_bytes, cudaMemcpyHostToDevice));
    if (half_rot && !e->d_rot) CU(upload(d_rot, rotation_table(2, 1)));
    const float2 *rotp = e->d_rot ? e->d_rot : d_rot;
    e->launches += launch_front_end(d_pk, d_x2, rotp, 1, half_rot ? 2 : 1, 1, e->sample_bits, 1, 0, e->stream);
    const float2 *sel_x2 = d_x2 + (half_rot ? kN : 0);
    e->launches += launch_fwd_fft(sel_x2, d_D, e->d_tables, 1, false, e->sm_count, e->stream);
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(e->stream));
    if (x2) CU(cudaMemcpy(x2, sel_x2, kN * sizeof(float2), cudaMemcpyDeviceToHost));
    if (D) CU(cudaMemcpy(D, d_D, kN * sizeof(float2), cudaMemcpyDeviceToHost));
    return ACQ_OK;
}

int acq_n_sats(const acq_engine *e) { return e ? (int)e->sats.size() : fail(ACQ_ERR_ARG, "engine is NULL"); }

int acq_get_params(const acq_engine *e, acq_params *p)
{
    if (!e || !p) return fail(ACQ_ERR_ARG, "NULL argument");
    *p = e->prm;
    return ACQ_OK;
}

int64_t acq_launch_count(const acq_engine *e) { return e ? e->launches : 0; }

int acq_plan_launch(int k_noncoh, int half_bin, int e1b, int64_t n_tiles, int sm_count, acq_launch_plan *out)
{
    if (!out || k_noncoh < 1 || sm_count < 1 || n_tiles < 1 || n_tiles > acq::kMaxTilesPerLaunch)
        return fail(ACQ_ERR_ARG, "acq_plan_launch: bad argument");
    memset(out, 0, sizeof *out);
    const int kind = e1b ? acq::search_kind_e1b(n_tiles, sm_count) : acq::search_kind_l1(k_noncoh, half_bin);
    out->kernel = kind;
    out->grid = acq::search_grid_ctas(n_tiles, kind, sm_count);
    out->claims = kind != acq::kSearchE1bCluster && acq::search_claims_tiles(n_tiles, out->grid);
    out->n_chunks = n_tiles;
    acq::search_chunk_lengths(&out->chunk_big, &out->chunk_mid);
    if (kind == acq::kSearchL1Cr) {
        acq::search_chunks(n_tiles, 2 * sm_count, &out->n_big, &out->n_mid);
        out->n_chunks = acq::search_chunk_count(n_tiles, 2 * sm_count);
    }
    return ACQ_OK;
}

int acq_set_profiling(acq_engine *e, int enable)
{
    if (!e) return fail(ACQ_ERR_ARG, "engine is NULL");
    DeviceGuard g(e->device);
    if (enable && !e->prof[0])
        for (cudaEvent_t &ev : e->prof) CU(cudaEventCreate(&ev));
    e->profiling = enable != 0;
    if (!enable) e->prof_valid = false;
    return ACQ_OK;
}

int acq_get_kernel_ms(acq_engine *e, float *out, int n_out)
{
    if (!e || !out || n_out < 4) return fail(ACQ_ERR_ARG, "bad argument");
    if (!e->prof_valid) return fail(ACQ_ERR_ARG, "no profiled search yet (call acq_set_profiling first)");
    DeviceGuard g(e->device);
    CU(cudaEventSynchronize(e->prof[4]));
    for (int i = 0; i < 4; i++) CU(cudaEventElapsedTime(&out[i], e->prof[i], e->prof[i + 1]));
    return ACQ_OK;
}

int acq_device_info(const acq_engine *e, int *device, int *sm_count, int *sm_clock_khz)
{
    if (!e) return fail(ACQ_ERR_ARG, "engine is NULL");
    if (device) *device = e->device;
    if (sm_count) *sm_count = e->sm_count;
    if (sm_clock_khz) *sm_clock_khz = e->sm_clock_khz;
    return ACQ_OK;
}

}  // extern "C"
