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
    // device-path ordering: an event behind the last acq_search_device; whatever touches the shared scratch next waits for it
    cudaEvent_t dev_done = nullptr;
    bool dev_pending = false;
    int64_t launches = 0;
    bool profiling = false, prof_valid = false;
    cudaEvent_t prof[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};

    // persistent device data
    float2 *d_tables = nullptr, *d_rot = nullptr, *d_C = nullptr, *d_Ep = nullptr;
    // per-call scratch (grown on demand)
    size_t cap_blocks = 0 /* spectrum rows */, cap_cells = 0, cap_rows = 0, cap_packed = 0;
    uint8_t *d_packed = nullptr;
    float2 *d_x2 = nullptr, *d_Dp = nullptr;
    acq_cell *d_cells = nullptr;
    acq_record *d_records = nullptr;
    unsigned *d_tile_ctr = nullptr;    // [4] claim counters [0,1] and done counters [2,3] of the C/A and the E1B search launch (SearchArgs::tile_ctr); zero between launches
    unsigned *d_ctas_done = nullptr;   // finished search CTAs of a small search (folded best-Doppler pick); zero between searches
    unsigned epoch = 0;                // search counter: value of the completion word
    // host path: pinned staging of small captures; records and the completion word in mapped pinned memory,
    // written by the search kernels themselves
    uint8_t *h_packed = nullptr;
    size_t cap_h_packed = 0;
    acq_record *h_records = nullptr, *dh_records = nullptr;  // host / device address of the same mapped buffer
    size_t cap_h_records = 0;
    unsigned *h_flag = nullptr, *dh_flag = nullptr;
    // selection: work list [n_slots] (C/A entries first, then E1B) and slot -> table index
    std::vector<int32_t> sel_cache;
    int sel_kind = -1;  // -1 none, 0 whole table, 1 one satellite, 2 uploaded list
    int n_l1 = 0, n_e1b = 0, n_slots = 0;
    const int2 *cur_work = nullptr;
    const int *cur_slot_sat = nullptr;
    int2 *d_work_full = nullptr, *d_work_single = nullptr, *d_work = nullptr;   // whole table / (s, 0) per s / uploaded
    int *d_sat_full = nullptr, *d_slot_sat = nullptr;                            // identity / uploaded
    int full_n_l1 = 0;
    size_t cap_slots = 0;
    // refinement (acq_refine): satellite types on the device, record/output scratch, shape of the last host-path search
    int *d_sat_type = nullptr;
    acq_record *d_ref_rec = nullptr;
    acq_fine *d_fine = nullptr;
    size_t cap_ref_rec = 0, cap_fine = 0;
    int last_captures = 0;  // 0: no search whose spectra are still on the device
    // shape of the most recent search of either path (acq_refine_device): captures (0: none whose spectra are still on
    // the device), slots, and its slot -> satellite map on the device
    int ref_captures = 0, ref_slots = 0;
    const int *ref_slot_sat = nullptr;
    int ref_n_l1 = 0, ref_n_e1b = 0;   // ... and its C/A and E1B slot counts (acq_profile_device)
    // peak-quality profile (acq_profile): row output scratch of the host form (its lag profiles get a buffer per call)
    acq_peak2 *d_peak2 = nullptr;
    size_t cap_peak2 = 0;
    // aided host search (acq_search_aided): Doppler centres staged in pinned memory, copied to the device with the capture
    int32_t *h_center = nullptr;
    size_t cap_h_center = 0;
    int *d_center = nullptr;
    size_t cap_center = 0;
    // coherent search (acq_search_coherent): sub-bin rotation table [F][16384] of each m_coh, built on first use
    float2 *d_rot_coh[ACQ_COH_MAX + 1] = {};
};

namespace {

using namespace acq;

// Build-time switches of the experiment variants (tools/build_variants.py); the product library defines none of
// them and reads no environment variable.
//   ACQ_FORCE_E1B_KERNEL=1|2 one-CTA / cluster form of the E1B search regardless of the tile count
#ifndef ACQ_FORCE_E1B_KERNEL
#define ACQ_FORCE_E1B_KERNEL 0
#endif
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

int free_engine(acq_engine *e)
{
    if (!e) return ACQ_OK;
    DeviceGuard g(e->device);
    if (e->stream) cudaStreamSynchronize(e->stream);
    if (e->dev_pending && e->dev_done) cudaEventSynchronize(e->dev_done);
    cudaFree(e->d_tables);
    cudaFree(e->d_rot);
    cudaFree(e->d_C);
    cudaFree(e->d_Ep);
    cudaFree(e->d_packed);
    cudaFree(e->d_x2);
    cudaFree(e->d_Dp);
    cudaFree(e->d_cells);
    cudaFree(e->d_records);
    cudaFree(e->d_ctas_done);
    cudaFree(e->d_tile_ctr);
    cudaFree(e->d_work_full);
    cudaFree(e->d_work_single);
    cudaFree(e->d_work);
    cudaFree(e->d_sat_full);
    cudaFree(e->d_slot_sat);
    cudaFree(e->d_sat_type);
    cudaFree(e->d_ref_rec);
    cudaFree(e->d_fine);
    cudaFree(e->d_peak2);
    cudaFree(e->d_center);
    for (float2 *r : e->d_rot_coh) cudaFree(r);
    if (e->h_center) cudaFreeHost(e->h_center);
    if (e->h_packed) cudaFreeHost(e->h_packed);
    if (e->h_records) cudaFreeHost(e->h_records);
    if (e->h_flag) cudaFreeHost(e->h_flag);
    if (e->done) cudaEventDestroy(e->done);
    if (e->dev_done) cudaEventDestroy(e->dev_done);
    for (cudaEvent_t ev : e->prof)
        if (ev) cudaEventDestroy(ev);
    if (e->stream) cudaStreamDestroy(e->stream);
    delete e;
    return ACQ_OK;
}

// Everything that is about to touch the shared scratch from the host (reallocation, synchronous copies) first
// drains the engine stream and the last device-path search.
int drain(acq_engine *e)
{
    CU(cudaStreamSynchronize(e->stream));
    if (e->dev_pending) {
        CU(cudaEventSynchronize(e->dev_done));
        e->dev_pending = false;
    }
    return ACQ_OK;
}

template <typename T>
int grow(acq_engine *e, T *&ptr, size_t &cap, size_t need_elems, bool zero = false)
{
    if (need_elems <= cap && ptr) return ACQ_OK;
    int rc = drain(e);
    if (rc) return rc;
    if (ptr) CU(cudaFree(ptr));
    ptr = nullptr;
    cap = 0;
    CU(cudaMalloc(&ptr, need_elems * sizeof(T)));
    if (zero) CU(cudaMemset(ptr, 0, need_elems * sizeof(T)));
    cap = need_elems;
    return ACQ_OK;
}

// n_dop: Doppler cells per row of this search (the engine's range, the window of an aided search, or the 1/M-bin grid of
// a coherent one); nvar: spectrum variants per block (e->nvar, or F of a coherent search)
int ensure_scratch(acq_engine *e, int n_captures, int n_slots, bool host_path, int n_dop, int nvar)
{
    const size_t blocks = (size_t)n_captures * e->prm.k_noncoh;
    const size_t spectra = blocks * nvar * e->n_shift;   // rows of x2 and of the capture spectra
    if (spectra > e->cap_blocks || !e->d_x2) {
        int rc = drain(e);  // changing scratch under an in-flight search is not allowed
        if (rc) return rc;
        if (e->d_x2) CU(cudaFree(e->d_x2));
        if (e->d_Dp) CU(cudaFree(e->d_Dp));
        e->d_x2 = e->d_Dp = nullptr;
        e->cap_blocks = 0;
        CU(cudaMalloc(&e->d_x2, spectra * kN * sizeof(float2)));
        CU(cudaMalloc(&e->d_Dp, spectra * kN * sizeof(float2)));
        e->cap_blocks = spectra;
    }
    const size_t rows = (size_t)n_captures * n_slots;
    int rc;
    if ((rc = grow(e, e->d_cells, e->cap_cells, rows * n_dop))) return rc;
    if (!host_path) return ACQ_OK;
    const size_t bytes = blocks * e->block_bytes;
    if ((rc = grow(e, e->d_packed, e->cap_packed, bytes))) return rc;
    if (bytes <= kStagePackedMax && bytes > e->cap_h_packed) {
        if ((rc = drain(e))) return rc;
        if (e->h_packed) CU(cudaFreeHost(e->h_packed));
        e->h_packed = nullptr;
        e->cap_h_packed = 0;
        CU(cudaHostAlloc(&e->h_packed, bytes, cudaHostAllocDefault));
        e->cap_h_packed = bytes;
    }
    if (rows <= (size_t)kHostRecordRowsMax) {
        if (rows > e->cap_h_records) {
            if ((rc = drain(e))) return rc;
            if (e->h_records) CU(cudaFreeHost(e->h_records));
            e->h_records = e->dh_records = nullptr;
            e->cap_h_records = 0;
            // sized for the tagged form a polling host reads (acq_record_tagged, 32 B); the plain 24-byte form fits too
            CU(cudaHostAlloc(&e->h_records, rows * sizeof(acq_record_tagged), cudaHostAllocMapped));
            memset(e->h_records, 0, rows * sizeof(acq_record_tagged));
            CU(cudaHostGetDevicePointer(&e->dh_records, e->h_records, 0));
            e->cap_h_records = rows;
        }
        return ACQ_OK;
    }
    return grow(e, e->d_records, e->cap_rows, rows);
}

// Split the selection into the 1 ms-window (Navstar/QZSS/SBAS) and E1B work lists.  The whole table and single
// satellites (what the literal SearchTask loop asks for, one satellite per capture) use lists built at acq_create;
// any other list is uploaded, which drains the engine first.
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
    if (n_sel <= 0) return fail(ACQ_ERR_ARG, "n_sel must be > 0 when sel is given");
    for (int i = 0; i < n_sel; i++)
        if (sel[i] < 0 || sel[i] >= n_sats)
            return fail(ACQ_ERR_ARG, "satellite index %d outside the table (0..%d)", sel[i], n_sats - 1);
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
    if ((size_t)n_sel > e->cap_slots) {
        if (e->d_work) CU(cudaFree(e->d_work));
        if (e->d_slot_sat) CU(cudaFree(e->d_slot_sat));
        e->d_work = nullptr;
        e->d_slot_sat = nullptr;
        e->cap_slots = 0;
        CU(cudaMalloc(&e->d_work, (size_t)n_sel * sizeof(int2)));
        CU(cudaMalloc(&e->d_slot_sat, (size_t)n_sel * sizeof(int)));
        e->cap_slots = (size_t)n_sel;
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

// Doppler cells per row: the engine's whole range, or the window of an aided search (center != NULL)
int row_dops(const acq_engine *e, const void *center, int half_width) { return center ? 2 * half_width + 1 : e->n_dop; }

// Coherent search of M = m_coh blocks per group: n_dop_c = M (n_dop - 1) + 1 cells per row (1/M of the engine's Doppler
// step), F = M (1 + half_bin) spectrum variants per block
int coh_dops(const acq_engine *e, int m_coh) { return m_coh * (e->n_dop - 1) + 1; }
int coh_variants(const acq_engine *e, int m_coh) { return m_coh * (1 + e->prm.half_bin); }
// Doppler cells per row of any search: a window (center != NULL) of either grid, else the coherent or the engine's range
int search_dops(const acq_engine *e, const void *center, int half_width, int m_coh)
{
    return (m_coh && !center) ? coh_dops(e, m_coh) : row_dops(e, center, half_width);
}

// Rotation table of the sub-bin variants, [F][16384]: row v = exp(-2 pi i (v / F) n / N), double precision rounded once.
// The angle is pi (a n) / (b N) with a / b = 2 v / F in lowest terms, so that the row v = F / 2 of an even F is formed by
// the same operations as the half-bin table of acq_create (pi n / N) and rounds to the same floats.
int ensure_coh_rot(acq_engine *e, int m_coh)
{
    if (e->d_rot_coh[m_coh]) return ACQ_OK;
    const int F = coh_variants(e, m_coh);
    const double pi = 3.14159265358979323846264338327950288;
    std::vector<float2> rot((size_t)F * kN);
    for (int v = 0; v < F; v++) {
        const int g = std::gcd(2 * v, F), a = 2 * v / g, b = F / g;
        for (int n = 0; n < kN; n++) {
            const double ang = pi * (double)((long long)a * n) / (double)((long long)b * kN);
            rot[(size_t)v * kN + n] = make_float2((float)cos(ang), (float)(-sin(ang)));
        }
    }
    float2 *d = nullptr;
    CU(cudaMalloc(&d, rot.size() * sizeof(float2)));
    const cudaError_t ce = cudaMemcpy(d, rot.data(), rot.size() * sizeof(float2), cudaMemcpyHostToDevice);
    if (ce != cudaSuccess) {
        cudaFree(d);
        return fail(ACQ_ERR_CUDA, "coherent rotation table: %s", cudaGetErrorString(ce));
    }
    e->d_rot_coh[m_coh] = d;
    return ACQ_OK;
}

int check_search_args(acq_engine *e, const void *packed, int n_captures, const void *out);

// The arguments of a coherent search, checked before anything touches the device: ACQ_ERR_ARG for the argument errors,
// ACQ_ERR_UNSUPPORTED for what the coherent search does not cover (E1B rows, code-Doppler engines, searches above the
// tile and spectrum-row bounds).  center != NULL: an aided coherent search, whose rows hold W = 2 half_width + 1 cells
// (W <= n_dop_c) rather than n_dop_c; check_coherent_aided_args has checked what needs no engine.
int check_coherent(acq_engine *e, const void *packed, int n_captures, const int32_t *sel, int n_sel, int m_coh,
                   const void *out, const int32_t *center = nullptr, int half_width = 0)
{
    if (!e) return fail(ACQ_ERR_ARG, "engine is NULL");
    if (m_coh < 1 || m_coh > ACQ_COH_MAX) return fail(ACQ_ERR_ARG, "m_coh=%d outside 1..%d", m_coh, ACQ_COH_MAX);
    int rc = check_search_args(e, packed, n_captures, out);
    if (rc) return rc;
    if (e->prm.k_noncoh % m_coh)
        return fail(ACQ_ERR_ARG, "k_noncoh=%d is not a multiple of m_coh=%d", e->prm.k_noncoh, m_coh);
    if (center && half_width > (coh_dops(e, m_coh) - 1) / 2)
        return fail(ACQ_ERR_ARG, "Doppler window W = 2*half_width+1 with half_width %d exceeds n_dop_c = %d", half_width,
                    coh_dops(e, m_coh));
    const int n_sats = (int)e->sats.size();
    if (sel && n_sel <= 0) return fail(ACQ_ERR_ARG, "n_sel must be > 0 when sel is given");
    const int n_slots = sel ? n_sel : n_sats;
    for (int i = 0; i < n_slots; i++) {
        const int s = sel ? sel[i] : i;
        if (s < 0 || s >= n_sats) return fail(ACQ_ERR_ARG, "satellite index %d outside the table (0..%d)", s, n_sats - 1);
    }
    if (e->prm.code_doppler)
        return fail(ACQ_ERR_UNSUPPORTED, "coherent search of a code_doppler engine is not implemented");
    for (int i = 0; i < n_slots; i++)
        if (e->sats[sel ? sel[i] : i].type == ACQ_E1B)
            return fail(ACQ_ERR_UNSUPPORTED, "coherent search of E1B rows is not implemented (satellite %d): E1B symbols "
                        "drift against the block edges", sel ? sel[i] : i);
    if ((long long)n_captures * e->prm.k_noncoh * coh_variants(e, m_coh) > (1 << 24))
        return fail(ACQ_ERR_UNSUPPORTED, "coherent search too large for one call (more than 2^24 capture spectra): split the captures");
    const int n_dop = center ? 2 * half_width + 1 : coh_dops(e, m_coh);
    if ((double)n_captures * (double)n_slots * (double)n_dop > (double)acq::kMaxTilesPerLaunch)
        return fail(ACQ_ERR_UNSUPPORTED, "coherent search too large for one call (more than 2^31 - 1 tiles): split the captures");
    return ACQ_OK;
}

// Enqueue front end + forward FFT + search (which ends in the best-Doppler pick) on `st` for captures already on the
// device.  records_dev: where the kernels write the records (device memory, or the device alias of mapped host memory);
// flag_dev: mapped completion word, or NULL.  center_dev: the rows' Doppler centres on the device (an aided search), or
// NULL for the whole range.  m_coh > 0: a coherent search (acq_search_coherent) of M = m_coh blocks per group, with
// center_dev its aided form (acq_search_coherent_aided: centres and half_width in the coherent grid's units).
int enqueue_search(acq_engine *e, const uint8_t *packed_dev, int n_captures, acq_record *records_dev, unsigned *flag_dev,
                   cudaStream_t st, const uint8_t *packed_host_arg = nullptr, const int *center_dev = nullptr,
                   int half_width = 0, int m_coh = 0)
{
    const int K = e->prm.k_noncoh;
    const int n_dop = search_dops(e, center_dev, half_width, m_coh);
    const int nvar = m_coh ? coh_variants(e, m_coh) : e->nvar;
    const int blocks = n_captures * K;
    const bool prof = e->profiling;
    if (e->dev_pending) CU(cudaStreamWaitEvent(st, e->dev_done, 0));  // a no-op on the stream that recorded it
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
        const float2 *rot = m_coh ? e->d_rot_coh[m_coh] + kN : e->d_rot;
        e->launches += launch_front_end(packed_dev, e->d_x2, rot, blocks, nvar, K, e->sample_bits, e->n_shift, e->smax, st);
        if (nvar > 2) e->launches += launch_coh_variants(e->d_x2, e->d_rot_coh[m_coh], blocks, nvar, K, st);
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
    a.dop_lo = e->prm.dop_lo * (m_coh ? m_coh : 1);
    a.dop_center = center_dev;
    a.half_width = half_width;
    a.dop_hi = e->prm.dop_hi * (m_coh ? m_coh : 1);
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
    // Cluster/DSMEM form of the E1B search when every tile can have a cluster of its own (one wave: 9 us per tile
    // against 12.5 us for the one-CTA form, measured) or when forced (variant builds).  With more tiles than that the
    // one-CTA-per-tile forms (k_search_e1b, k_search_e1b_multi for non-coherent sums) have ~2.9x the throughput.
    const bool e1b_cluster = ACQ_FORCE_E1B_KERNEL == 2 || (ACQ_FORCE_E1B_KERNEL == 0 && tiles_e1b <= e->sm_count / 4);
    a.ctas_done = e->d_ctas_done;
    a.ctas_total = fold ? (unsigned)((m_coh ? coh_grid_ctas(tiles_l1, e->sm_count)
                                            : search_grid_ctas(tiles_l1, search_kind_l1(K, e->prm.half_bin), e->sm_count)) +
                                     search_grid_ctas(tiles_e1b, e1b_cluster ? kSearchE1bCluster : kSearchE1b, e->sm_count))
                        : 0u;
    a.wait_prior = 1;
    if (m_coh && e->n_l1 > 0) {   // the selection holds no E1B row (check_coherent)
        a.work = e->cur_work;
        a.n_work = e->n_l1;
        a.n_tiles = tiles_l1;
        a.tile_ctr = e->d_tile_ctr;
        e->launches += launch_search_coh(CohSearchArgs(a, m_coh), e->sm_count, st, pdl);
    } else if (e->n_l1 > 0) {
        a.work = e->cur_work;
        a.n_work = e->n_l1;
        a.n_tiles = tiles_l1;
        a.tile_ctr = e->d_tile_ctr;
        e->launches += launch_search(a, false, e->sm_count, st, pdl);
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
        if (e1b_cluster) e->launches += launch_search_e1b_cluster(a, e->sm_count, st, pdl);
        else e->launches += launch_search(a, true, e->sm_count, st, pdl);
    }
    if (prof) CU(cudaEventRecord(e->prof[3], st));
    const PickDop pd{a.dop_lo, center_dev, half_width, a.dop_hi};
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

int check_search_args(acq_engine *e, const void *packed, int n_captures, const void *out)
{
    if (!e) return fail(ACQ_ERR_ARG, "engine is NULL");
    if (!packed || !out) return fail(ACQ_ERR_ARG, "packed/out must not be NULL");
    if (n_captures <= 0) return fail(ACQ_ERR_ARG, "n_captures must be > 0 (got %d)", n_captures);
    if ((long long)n_captures * e->prm.k_noncoh * e->n_shift > (1 << 24)) return fail(ACQ_ERR_ARG, "too many capture blocks");
    if (e->pending) return fail(ACQ_ERR_ARG, "a submitted search is still pending: call acq_wait first");
    return ACQ_OK;
}

// after set_selection: a search kernel launch indexes its tiles with 32 bits (and four units per tile with 64)
int check_tile_count(acq_engine *e, int n_captures, int n_dop)
{
    if ((double)n_captures * (double)e->n_slots * (double)n_dop > (double)acq::kMaxTilesPerLaunch)
        return fail(ACQ_ERR_UNSUPPORTED, "search too large for one call (more than 2^31 - 1 tiles): split the captures");
    return ACQ_OK;
}

// Largest Doppler range an engine can have: |index| <= 4094 half-bins (acq_create: at most 2048 bins either side).
constexpr int kMaxHalfWidth = 4094;

// Arguments of an aided search that need no engine come first, so that they are reported whatever the engine.
int check_aided_args(acq_engine *e, const int32_t *dop_center, int half_width)
{
    if (!dop_center) return fail(ACQ_ERR_ARG, "dop_center is NULL");
    if (half_width < 0) return fail(ACQ_ERR_ARG, "half_width must be >= 0 (got %d)", half_width);
    if (half_width > kMaxHalfWidth)
        return fail(ACQ_ERR_ARG, "Doppler window W = 2*half_width+1 with half_width %d exceeds n_dop of any engine", half_width);
    if (!e) return fail(ACQ_ERR_ARG, "engine is NULL");
    if (2 * half_width + 1 > e->n_dop)
        return fail(ACQ_ERR_ARG, "Doppler window W = 2*half_width+1 = %d exceeds n_dop = %d", 2 * half_width + 1, e->n_dop);
    return ACQ_OK;
}

// Arguments of an aided coherent search that need no engine come first, as in check_aided_args.
int check_coherent_aided_args(acq_engine *e, const int32_t *dop_center, int half_width, int m_coh)
{
    if (!dop_center) return fail(ACQ_ERR_ARG, "dop_center is NULL");
    if (half_width < 0) return fail(ACQ_ERR_ARG, "half_width must be >= 0 (got %d)", half_width);
    if (m_coh < 1 || m_coh > ACQ_COH_MAX) return fail(ACQ_ERR_ARG, "m_coh=%d outside 1..%d", m_coh, ACQ_COH_MAX);
    if (half_width > ACQ_COH_MAX * kMaxHalfWidth)
        return fail(ACQ_ERR_ARG, "Doppler window W = 2*half_width+1 with half_width %d exceeds n_dop_c of any engine", half_width);
    if (!e) return fail(ACQ_ERR_ARG, "engine is NULL");
    return ACQ_OK;
}

// Wait for a host-polled search and collect its records: k_pick_small writes every record into mapped memory as two
// 16-byte halves that each end in the search's epoch (acq_record_tagged), so a half whose tag matches has arrived whole.
// The stream is queried now and then so that a failed launch cannot hang the caller; the mapped word *h_flag is only
// ever written to report that the pick gave up (0xffffffff).
int poll_records(acq_engine *e, acq_record *out, size_t rows)
{
    const volatile acq_record_tagged *h = reinterpret_cast<const volatile acq_record_tagged *>(e->h_records);
    const unsigned epoch = e->epoch;
    unsigned spins = 0;
    for (size_t i = 0; i < rows; i++) {
        while (h[i].tag0 != epoch || h[i].tag1 != epoch) {
            if ((++spins & 0x3ff) == 0) {
                if (*(volatile unsigned *)e->h_flag == 0xffffffffu) {
                    *e->h_flag = 0;
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

// After a search of either path is enqueued: the shape acq_refine_device and acq_profile_device check their call and
// their records against.
void set_refine_shape(acq_engine *e, int n_captures)
{
    e->ref_captures = n_captures;
    e->ref_slots = e->n_slots;
    e->ref_slot_sat = e->cur_slot_sat;
    e->ref_n_l1 = e->n_l1;
    e->ref_n_e1b = e->n_e1b;
}

int enqueue_refine(acq_engine *e, const acq_record *rec_dev, int n_records, int flags, acq_fine *out_dev,
                   const int *slot_sat, int n_slots, cudaStream_t st)
{
    e->launches += launch_refine(e->d_Dp, e->d_Ep, rec_dev, e->d_sat_type, slot_sat, out_dev, n_records, n_slots,
                                 e->prm.k_noncoh, e->nvar, e->prm.half_bin, e->ext_len, e->Q, e->n_shift, e->smax,
                                 e->cd_div, (int)e->sats.size(), e->prm.dop_lo, e->prm.dop_hi, e->prm.thr_l1,
                                 e->prm.thr_e1b, flags, st);
    CU(cudaGetLastError());
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

int enqueue_profile(acq_engine *e, const acq_record *rec_dev, int n_records, int flags, int excl, acq_peak2 *out_dev,
                    float *profile_dev, const int *slot_sat, int n_slots, int n_l1, int n_e1b, cudaStream_t st)
{
    e->launches += launch_profile(e->d_Dp, e->d_Ep, e->d_tables, rec_dev, e->d_sat_type, slot_sat, out_dev, profile_dev,
                                  n_records, n_slots, n_l1, n_e1b, e->prm.k_noncoh, e->nvar, e->prm.half_bin, e->ext_len, e->Q,
                                  e->n_shift, e->smax, e->cd_div, (int)e->sats.size(), e->prm.dop_lo, e->prm.dop_hi,
                                  e->prm.thr_l1, e->prm.thr_e1b, flags, excl, st);
    CU(cudaGetLastError());
    return ACQ_OK;
}

// center (HOST, one per row) and half_width: an aided search (acq_search_aided), or NULL for the whole range
// m_coh > 0: a coherent search (acq_search_coherent, or with center acq_search_coherent_aided), its arguments already
// checked by check_coherent
int search_host(acq_engine *e, const uint8_t *packed, int n_captures, const int32_t *sel, int n_sel, acq_record *out,
                acq_cell *grid, bool sync, const int32_t *center = nullptr, int half_width = 0, int m_coh = 0)
{
    int rc = check_search_args(e, packed, n_captures, out);
    if (rc) return rc;
    DeviceGuard g(e->device);
    e->last_captures = 0;  // until this search is enqueued, there are no spectra acq_refine could use
    e->ref_captures = 0;
    const int n_dop = search_dops(e, center, half_width, m_coh);
    if ((rc = set_selection(e, sel, n_sel))) return rc;
    if ((rc = check_tile_count(e, n_captures, n_dop))) return rc;
    if ((rc = ensure_scratch(e, n_captures, e->n_slots, true, n_dop, m_coh ? coh_variants(e, m_coh) : e->nvar))) return rc;
    if (m_coh && (rc = ensure_coh_rot(e, m_coh))) return rc;
    const size_t bytes = (size_t)n_captures * e->prm.k_noncoh * e->block_bytes;
    const size_t rows = (size_t)n_captures * e->n_slots;
    if (center) {
        if ((rc = grow(e, e->d_center, e->cap_center, rows))) return rc;
        if (rows > e->cap_h_center) {
            if ((rc = drain(e))) return rc;
            if (e->h_center) CU(cudaFreeHost(e->h_center));
            e->h_center = nullptr;
            e->cap_h_center = 0;
            CU(cudaHostAlloc(&e->h_center, rows * sizeof(int32_t), cudaHostAllocDefault));
            e->cap_h_center = rows;
        }
    }
    const bool host_records = rows <= (size_t)kHostRecordRowsMax;
    const long long tiles_total = (long long)rows * n_dop * e->prm.k_noncoh;
    const bool poll = host_records && sync && !grid && !e->profiling && tiles_total <= 64LL * e->sm_count;
    // The reference's own search -- one 1-bit block (gps/search.cpp:389-411) -- hands its 8 KiB to the front end as a
    // kernel argument: the launch carries the bytes, nothing is staged or copied ahead of the first kernel.
    const bool as_arg = ACQ_ARG_INPUT && !m_coh && n_captures == 1 && e->prm.k_noncoh == 1 && e->sample_bits == 1 &&
                        bytes == (size_t)ACQ_BLOCK_BYTES;
    const uint8_t *src = packed;
    if (!as_arg) {
        if (bytes <= kStagePackedMax) {
            memcpy(e->h_packed, packed, bytes);
            src = e->h_packed;
        }
        CU(cudaMemcpyAsync(e->d_packed, src, bytes, cudaMemcpyHostToDevice, e->stream));
    }
    if (center) {   // from pinned memory: an asynchronous copy node ahead of the front end, even when the capture rides as an argument
        memcpy(e->h_center, center, rows * sizeof(int32_t));
        CU(cudaMemcpyAsync(e->d_center, e->h_center, rows * sizeof(int32_t), cudaMemcpyHostToDevice, e->stream));
    }
    if ((rc = enqueue_search(e, e->d_packed, n_captures, host_records ? e->dh_records : e->d_records,
                             poll ? e->dh_flag : nullptr, e->stream, as_arg ? packed : nullptr, center ? e->d_center : nullptr,
                             half_width, m_coh)))
        return rc;
    if (!m_coh) {   // a coherent search leaves spectra that refinement and profile cannot read
        e->last_captures = n_captures;
        set_refine_shape(e, n_captures);
    }
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
        if (host_records) memcpy(out, e->h_records, rows * sizeof(acq_record));
    }
    e->dev_pending = false;  // this search was ordered behind the last device-path search, so that one is complete too
    return ACQ_OK;
}

// completion of an acq_submit: records that the kernels left in the mapped buffer go to the caller's array
void finish_pending(acq_engine *e)
{
    if (e->pending_rows > 0 && e->pending_out)
        memcpy(e->pending_out, e->h_records, (size_t)e->pending_rows * sizeof(acq_record));
    e->pending = false;
    e->pending_rows = 0;
    e->pending_out = nullptr;
}

// acq_search_device and acq_search_aided_device (center_dev != NULL); with m_coh > 0 their coherent forms
int search_device(acq_engine *e, const uint8_t *packed_dev, int n_captures, const int32_t *sel, int n_sel,
                  acq_record *out_dev, void *stream, const int *center_dev = nullptr, int half_width = 0, int m_coh = 0)
{
    int rc = check_search_args(e, packed_dev, n_captures, out_dev);
    if (rc) return rc;
    if (((uintptr_t)packed_dev & 15) != 0)
        return fail(ACQ_ERR_ARG, "packed_dev must be 16-byte aligned (the front end stages it with bulk async copies)");
    DeviceGuard g(e->device);
    e->last_captures = 0;  // spectra now belong to a search on the caller's stream: acq_refine does not apply
    e->ref_captures = 0;   // ... and acq_refine_device applies once this search is enqueued
    const int n_dop = search_dops(e, center_dev, half_width, m_coh);
    if ((rc = set_selection(e, sel, n_sel))) return rc;
    if ((rc = check_tile_count(e, n_captures, n_dop))) return rc;
    if ((rc = ensure_scratch(e, n_captures, e->n_slots, false, n_dop, m_coh ? coh_variants(e, m_coh) : e->nvar))) return rc;
    if (m_coh && (rc = ensure_coh_rot(e, m_coh))) return rc;
    cudaStream_t st = stream ? (cudaStream_t)stream : e->stream;
    if ((rc = enqueue_search(e, packed_dev, n_captures, out_dev, nullptr, st, nullptr, center_dev, half_width, m_coh))) return rc;
    if (!m_coh) set_refine_shape(e, n_captures);
    if (st != e->stream) {  // whatever uses the engine's scratch next (any stream, or the host) waits for this search
        CU(cudaEventRecord(e->dev_done, st));
        e->dev_pending = true;
    }
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
    acq_engine *e = new acq_engine;
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

#define CUE(call)                                                                                   \
    do {                                                                                            \
        cudaError_t _e = (call);                                                                    \
        if (_e != cudaSuccess) {                                                                    \
            fail(ACQ_ERR_CUDA, "%s:%d %s: %s", __FILE__, __LINE__, #call, cudaGetErrorString(_e)); \
            free_engine(e);                                                                         \
            return ACQ_ERR_CUDA;                                                                    \
        }                                                                                           \
    } while (0)

    CUE(cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking));
    CUE(cudaEventCreateWithFlags(&e->done, cudaEventDisableTiming));
    CUE(cudaEventCreateWithFlags(&e->dev_done, cudaEventDisableTiming));
    CUE(search_kernels_configure());
    // completion counter of small searches, mapped completion word
    CUE(cudaMalloc(&e->d_ctas_done, sizeof(unsigned)));
    CUE(cudaMemset(e->d_ctas_done, 0, sizeof(unsigned)));
    CUE(cudaMalloc(&e->d_tile_ctr, 4 * sizeof(unsigned)));
    CUE(cudaMemset(e->d_tile_ctr, 0, 4 * sizeof(unsigned)));
    CUE(cudaHostAlloc(&e->h_flag, sizeof(unsigned), cudaHostAllocMapped));
    *e->h_flag = 0;
    CUE(cudaHostGetDevicePointer(&e->dh_flag, e->h_flag, 0));
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
        CUE(cudaMalloc(&e->d_work_full, n_sats * sizeof(int2)));
        CUE(cudaMalloc(&e->d_work_single, n_sats * sizeof(int2)));
        CUE(cudaMalloc(&e->d_sat_full, n_sats * sizeof(int)));
        CUE(cudaMemcpy(e->d_work_full, full.data(), n_sats * sizeof(int2), cudaMemcpyHostToDevice));
        CUE(cudaMemcpy(e->d_work_single, single.data(), n_sats * sizeof(int2), cudaMemcpyHostToDevice));
        CUE(cudaMemcpy(e->d_sat_full, ident.data(), n_sats * sizeof(int), cudaMemcpyHostToDevice));
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
    CUE(launch_tables_init(cC, hb));
    CUE(cudaMalloc(&e->d_tables, tables.size() * sizeof(float2)));
    CUE(cudaMemcpy(e->d_tables, tables.data(), tables.size() * sizeof(float2), cudaMemcpyHostToDevice));
    {
        std::vector<int> types(n_sats);
        for (int i = 0; i < n_sats; i++) types[i] = sats[i].type;
        CUE(cudaMalloc(&e->d_sat_type, n_sats * sizeof(int)));
        CUE(cudaMemcpy(e->d_sat_type, types.data(), n_sats * sizeof(int), cudaMemcpyHostToDevice));
    }
    if (e->nvar == 2) {
        const double pi = 3.14159265358979323846264338327950288;
        std::vector<float2> rot(kN);
        for (int n = 0; n < kN; n++) {
            const double a = pi * (double)n / (double)kN;
            rot[n] = make_float2((float)cos(a), (float)(-sin(a)));
        }
        CUE(cudaMalloc(&e->d_rot, kN * sizeof(float2)));
        CUE(cudaMemcpy(e->d_rot, rot.data(), kN * sizeof(float2), cudaMemcpyHostToDevice));
    }

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
    uint32_t *d_chips = nullptr;
    int *d_clb = nullptr;
    float2 *d_x1 = nullptr, *d_x2 = nullptr;
    cudaError_t ce = cudaSuccess;
    do {
        if ((ce = cudaMalloc(&d_chips, chips.size() * sizeof(uint32_t)))) break;
        if ((ce = cudaMalloc(&d_clb, codelen_boc.size() * sizeof(int)))) break;
        if ((ce = cudaMalloc(&d_x1, (size_t)n_sats * 32768 * sizeof(float2)))) break;
        if ((ce = cudaMalloc(&d_x2, (size_t)n_sats * kN * sizeof(float2)))) break;
        if ((ce = cudaMalloc(&e->d_C, (size_t)n_sats * kN * sizeof(float2)))) break;
        if ((ce = cudaMalloc(&e->d_Ep, (size_t)n_sats * 4 * e->ext_len * sizeof(float2)))) break;
        if ((ce = cudaMemcpy(d_chips, chips.data(), chips.size() * sizeof(uint32_t), cudaMemcpyHostToDevice))) break;
        if ((ce = cudaMemcpy(d_clb, codelen_boc.data(), codelen_boc.size() * sizeof(int), cudaMemcpyHostToDevice)))
            break;
        e->launches += launch_hb1_code(d_chips, d_clb, d_x1, n_sats, e->stream);
        e->launches += launch_hb2(d_x1, d_x2, nullptr, n_sats, 1, 1, e->stream);
        e->launches += launch_fwd_fft(d_x2, e->d_C, e->d_tables, n_sats, false, e->sm_count, e->stream);
        e->launches += launch_build_ext(e->d_C, e->d_Ep, n_sats, e->Q, e->ext_len, prm.wrap_mode, e->stream);
        if ((ce = cudaGetLastError())) break;
        ce = cudaStreamSynchronize(e->stream);
    } while (0);
    cudaFree(d_chips);
    cudaFree(d_clb);
    cudaFree(d_x1);
    cudaFree(d_x2);
    CUE(ce);
#undef CUE
    *out = e;
    return ACQ_OK;
}

int acq_destroy(acq_engine *e) { return free_engine(e); }

int acq_search(acq_engine *e, const uint8_t *packed, int n_captures, const int32_t *sel, int n_sel, acq_record *out)
{
    return search_host(e, packed, n_captures, sel, n_sel, out, nullptr, true);
}

int acq_search_grid(acq_engine *e, const uint8_t *packed, int n_captures, const int32_t *sel, int n_sel,
                    acq_record *out, acq_cell *grid)
{
    if (!grid) return fail(ACQ_ERR_ARG, "grid is NULL");
    return search_host(e, packed, n_captures, sel, n_sel, out, grid, true);
}

int acq_search_aided(acq_engine *e, const uint8_t *packed, int n_captures, const int32_t *sel, int n_sel,
                     const int32_t *dop_center, int half_width, acq_record *out, acq_cell *grid)
{
    const int rc = check_aided_args(e, dop_center, half_width);
    if (rc) return rc;
    return search_host(e, packed, n_captures, sel, n_sel, out, grid, true, dop_center, half_width);
}

int acq_search_device(acq_engine *e, const uint8_t *packed_dev, int n_captures, const int32_t *sel, int n_sel,
                      acq_record *out_dev, void *stream)
{
    return search_device(e, packed_dev, n_captures, sel, n_sel, out_dev, stream);
}

int acq_search_aided_device(acq_engine *e, const uint8_t *packed_dev, int n_captures, const int32_t *sel, int n_sel,
                            const int32_t *dop_center_dev, int half_width, acq_record *out_dev, void *stream)
{
    const int rc = check_aided_args(e, dop_center_dev, half_width);
    if (rc) return rc;
    return search_device(e, packed_dev, n_captures, sel, n_sel, out_dev, stream, dop_center_dev, half_width);
}

int acq_search_coherent(acq_engine *e, const uint8_t *packed, int n_captures, const int32_t *sel, int n_sel, int m_coh,
                        acq_record *out, acq_cell *grid)
{
    const int rc = check_coherent(e, packed, n_captures, sel, n_sel, m_coh, out);
    if (rc) return rc;
    return search_host(e, packed, n_captures, sel, n_sel, out, grid, true, nullptr, 0, m_coh);
}

int acq_search_coherent_device(acq_engine *e, const uint8_t *packed_dev, int n_captures, const int32_t *sel, int n_sel,
                               int m_coh, acq_record *out_dev, void *stream)
{
    const int rc = check_coherent(e, packed_dev, n_captures, sel, n_sel, m_coh, out_dev);
    if (rc) return rc;
    return search_device(e, packed_dev, n_captures, sel, n_sel, out_dev, stream, nullptr, 0, m_coh);
}

int acq_search_coherent_aided(acq_engine *e, const uint8_t *packed, int n_captures, const int32_t *sel, int n_sel,
                              int m_coh, const int32_t *dop_center, int half_width, acq_record *out, acq_cell *grid)
{
    int rc = check_coherent_aided_args(e, dop_center, half_width, m_coh);
    if (rc || (rc = check_coherent(e, packed, n_captures, sel, n_sel, m_coh, out, dop_center, half_width))) return rc;
    return search_host(e, packed, n_captures, sel, n_sel, out, grid, true, dop_center, half_width, m_coh);
}

int acq_search_coherent_aided_device(acq_engine *e, const uint8_t *packed_dev, int n_captures, const int32_t *sel,
                                     int n_sel, int m_coh, const int32_t *dop_center_dev, int half_width,
                                     acq_record *out_dev, void *stream)
{
    int rc = check_coherent_aided_args(e, dop_center_dev, half_width, m_coh);
    if (rc || (rc = check_coherent(e, packed_dev, n_captures, sel, n_sel, m_coh, out_dev, dop_center_dev, half_width)))
        return rc;
    return search_device(e, packed_dev, n_captures, sel, n_sel, out_dev, stream, dop_center_dev, half_width, m_coh);
}

int acq_submit(acq_engine *e, const uint8_t *packed, int n_captures, const int32_t *sel, int n_sel, acq_record *out)
{
    return search_host(e, packed, n_captures, sel, n_sel, out, nullptr, false);
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
    if (e->pending) return fail(ACQ_ERR_ARG, "a submitted search is still pending: call acq_wait first");
    if (e->last_captures <= 0) return fail(ACQ_ERR_ARG, "no completed host-path search to refine");
    const long long rows = (long long)e->last_captures * e->n_slots;
    if (n_records != rows)
        return fail(ACQ_ERR_ARG, "n_records=%d but the last search produced %lld records", n_records, rows);
    for (int i = 0; i < n_records; i++) {
        const acq_record &r = rec[i];
        if (r.sat != e->sel_cache[i % e->n_slots])
            return fail(ACQ_ERR_ARG, "record %d: sat %d is not the satellite searched in that slot", i, r.sat);
        const int L = (e->sats[r.sat].type == ACQ_E1B) ? ACQ_LAGS_E1B : ACQ_LAGS_L1;
        if (r.lag < 0 || r.lag >= L) return fail(ACQ_ERR_ARG, "record %d: lag %d outside 0..%d", i, r.lag, L - 1);
        // a row that never exceeded snr 0 carries dop 0 (k_best_dop), which may lie outside an asymmetric range
        if ((r.dop < e->prm.dop_lo || r.dop > e->prm.dop_hi) && !(r.dop == 0 && r.snr == 0.0f))
            return fail(ACQ_ERR_ARG, "record %d: Doppler index %d outside %d..%d", i, r.dop, e->prm.dop_lo, e->prm.dop_hi);
    }
    DeviceGuard g(e->device);
    int rc = grow(e, e->d_ref_rec, e->cap_ref_rec, (size_t)n_records);
    if (rc) return rc;
    if ((rc = grow(e, e->d_fine, e->cap_fine, (size_t)n_records))) return rc;
    CU(cudaMemcpyAsync(e->d_ref_rec, rec, (size_t)n_records * sizeof(acq_record), cudaMemcpyHostToDevice, e->stream));
    // the records are checked above, so the kernel's own checks pass every row
    if ((rc = enqueue_refine(e, e->d_ref_rec, n_records, 0, e->d_fine, e->cur_slot_sat, e->n_slots, e->stream))) return rc;
    CU(cudaMemcpyAsync(out, e->d_fine, (size_t)n_records * sizeof(acq_fine), cudaMemcpyDeviceToHost, e->stream));
    CU(cudaStreamSynchronize(e->stream));
    return ACQ_OK;
}

int acq_refine_device(acq_engine *e, const acq_record *rec_dev, int n_records, int flags, acq_fine *out_dev, void *stream)
{
    if (!e) return fail(ACQ_ERR_ARG, "engine is NULL");
    if (!rec_dev || !out_dev) return fail(ACQ_ERR_ARG, "rec_dev/out_dev must not be NULL");
    if (flags & ~ACQ_REFINE_DETECTED) return fail(ACQ_ERR_ARG, "unknown flag bits 0x%x", (unsigned)(flags & ~ACQ_REFINE_DETECTED));
    if (e->ref_captures <= 0) return fail(ACQ_ERR_ARG, "no search whose spectra are still on the device to refine");
    if (e->pending) return fail(ACQ_ERR_ARG, "a submitted search is still pending: call acq_wait first");
    const long long rows = (long long)e->ref_captures * e->ref_slots;
    if (n_records != rows)
        return fail(ACQ_ERR_ARG, "n_records=%d but the last search produced %lld records", n_records, rows);
    if (((uintptr_t)out_dev & 15) != 0) return fail(ACQ_ERR_ARG, "out_dev must be 16-byte aligned (one 16-byte store per row)");
    if (((uintptr_t)rec_dev & 3) != 0) return fail(ACQ_ERR_ARG, "rec_dev must be 4-byte aligned");
    DeviceGuard g(e->device);
    cudaStream_t st = stream ? (cudaStream_t)stream : e->stream;
    // after the search that left the spectra: a device-path search on another stream is behind dev_done, anything
    // else on the engine stream
    if (e->dev_pending) CU(cudaStreamWaitEvent(st, e->dev_done, 0));
    if (st != e->stream) {
        CU(cudaEventRecord(e->dev_done, e->stream));
        CU(cudaStreamWaitEvent(st, e->dev_done, 0));
    }
    int rc = enqueue_refine(e, rec_dev, n_records, flags, out_dev, e->ref_slot_sat, e->ref_slots, st);
    if (rc) return rc;
    if (st != e->stream) {  // the next search overwrites the spectra: whatever touches the scratch next waits for this
        CU(cudaEventRecord(e->dev_done, st));
        e->dev_pending = true;
    }
    return ACQ_OK;
}

int acq_profile(acq_engine *e, const acq_record *rec, int n_records, int excl, acq_peak2 *out, float *profile)
{
    if (!e) return fail(ACQ_ERR_ARG, "engine is NULL");
    if (!rec || !out) return fail(ACQ_ERR_ARG, "rec/out must not be NULL");
    if (excl < 0) return fail(ACQ_ERR_ARG, "excl must be >= 0 (got %d)", excl);
    if (e->pending) return fail(ACQ_ERR_ARG, "a submitted search is still pending: call acq_wait first");
    if (e->last_captures <= 0) return fail(ACQ_ERR_ARG, "no completed host-path search to profile");
    const long long rows = (long long)e->last_captures * e->n_slots;
    if (n_records != rows)
        return fail(ACQ_ERR_ARG, "n_records=%d but the last search produced %lld records", n_records, rows);
    int rc = check_excl(excl, e->n_l1);
    if (rc) return rc;
    for (int i = 0; i < n_records; i++) {   // acq_refine's checks
        const acq_record &r = rec[i];
        if (r.sat != e->sel_cache[i % e->n_slots])
            return fail(ACQ_ERR_ARG, "record %d: sat %d is not the satellite searched in that slot", i, r.sat);
        const int L = (e->sats[r.sat].type == ACQ_E1B) ? ACQ_LAGS_E1B : ACQ_LAGS_L1;
        if (r.lag < 0 || r.lag >= L) return fail(ACQ_ERR_ARG, "record %d: lag %d outside 0..%d", i, r.lag, L - 1);
        if ((r.dop < e->prm.dop_lo || r.dop > e->prm.dop_hi) && !(r.dop == 0 && r.snr == 0.0f))
            return fail(ACQ_ERR_ARG, "record %d: Doppler index %d outside %d..%d", i, r.dop, e->prm.dop_lo, e->prm.dop_hi);
    }
    DeviceGuard g(e->device);
    const size_t n_prof = (size_t)e->last_captures * profile_capture_len(e->n_l1, e->n_e1b);
    if ((rc = grow(e, e->d_ref_rec, e->cap_ref_rec, (size_t)n_records))) return rc;
    if ((rc = grow(e, e->d_peak2, e->cap_peak2, (size_t)n_records))) return rc;
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
    if ((rc = enqueue_profile(e, e->d_ref_rec, n_records, 0, excl, e->d_peak2, d_prof.p,
                              e->cur_slot_sat, e->n_slots, e->n_l1, e->n_e1b, e->stream)))
        return rc;
    CU(cudaMemcpyAsync(out, e->d_peak2, (size_t)n_records * sizeof(acq_peak2), cudaMemcpyDeviceToHost, e->stream));
    if (profile) CU(cudaMemcpyAsync(profile, d_prof.p, n_prof * sizeof(float), cudaMemcpyDeviceToHost, e->stream));
    CU(cudaStreamSynchronize(e->stream));
    return ACQ_OK;
}

int acq_profile_device(acq_engine *e, const acq_record *rec_dev, int n_records, int flags, int excl, acq_peak2 *out_dev,
                       float *profile_dev, void *stream)
{
    if (!e) return fail(ACQ_ERR_ARG, "engine is NULL");
    if (!rec_dev || !out_dev) return fail(ACQ_ERR_ARG, "rec_dev/out_dev must not be NULL");
    if (flags & ~ACQ_PROFILE_DETECTED) return fail(ACQ_ERR_ARG, "unknown flag bits 0x%x", (unsigned)(flags & ~ACQ_PROFILE_DETECTED));
    if (excl < 0) return fail(ACQ_ERR_ARG, "excl must be >= 0 (got %d)", excl);
    if (e->ref_captures <= 0) return fail(ACQ_ERR_ARG, "no search whose spectra are still on the device to profile");
    if (e->pending) return fail(ACQ_ERR_ARG, "a submitted search is still pending: call acq_wait first");
    const long long rows = (long long)e->ref_captures * e->ref_slots;
    if (n_records != rows)
        return fail(ACQ_ERR_ARG, "n_records=%d but the last search produced %lld records", n_records, rows);
    int rc = check_excl(excl, e->ref_n_l1);
    if (rc) return rc;
    if (((uintptr_t)out_dev & 15) != 0) return fail(ACQ_ERR_ARG, "out_dev must be 16-byte aligned (one 16-byte store per row)");
    if (((uintptr_t)rec_dev & 3) != 0) return fail(ACQ_ERR_ARG, "rec_dev must be 4-byte aligned");
    if (((uintptr_t)profile_dev & 3) != 0) return fail(ACQ_ERR_ARG, "profile_dev must be 4-byte aligned");
    DeviceGuard g(e->device);
    cudaStream_t st = stream ? (cudaStream_t)stream : e->stream;
    // ordered as acq_refine_device: after the search that left the spectra, before the next one
    if (e->dev_pending) CU(cudaStreamWaitEvent(st, e->dev_done, 0));
    if (st != e->stream) {
        CU(cudaEventRecord(e->dev_done, e->stream));
        CU(cudaStreamWaitEvent(st, e->dev_done, 0));
    }
    if ((rc = enqueue_profile(e, rec_dev, n_records, flags, excl, out_dev, profile_dev, e->ref_slot_sat, e->ref_slots,
                              e->ref_n_l1, e->ref_n_e1b, st)))
        return rc;
    if (st != e->stream) {
        CU(cudaEventRecord(e->dev_done, st));
        e->dev_pending = true;
    }
    return ACQ_OK;
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
    uint8_t *d_pk = nullptr;
    float2 *d_x2 = nullptr, *d_D = nullptr, *d_rot = nullptr;
    std::vector<float2> rot;
    int rc = ACQ_OK;
    cudaError_t ce = cudaSuccess;
    do {
        if ((ce = cudaMalloc(&d_pk, e->block_bytes))) break;
        if ((ce = cudaMalloc(&d_x2, 2 * kN * sizeof(float2)))) break;
        if ((ce = cudaMalloc(&d_D, kN * sizeof(float2)))) break;
        if ((ce = cudaMemcpy(d_pk, packed, e->block_bytes, cudaMemcpyHostToDevice))) break;
        const float2 *rotp = e->d_rot;
        if (half_rot && !rotp) {
            const double pi = 3.14159265358979323846264338327950288;
            rot.resize(kN);
            for (int n = 0; n < kN; n++) {
                const double a = pi * (double)n / (double)kN;
                rot[n] = make_float2((float)cos(a), (float)(-sin(a)));
            }
            if ((ce = cudaMalloc(&d_rot, kN * sizeof(float2)))) break;
            if ((ce = cudaMemcpy(d_rot, rot.data(), kN * sizeof(float2), cudaMemcpyHostToDevice))) break;
            rotp = d_rot;
        }
        e->launches += launch_front_end(d_pk, d_x2, rotp, 1, half_rot ? 2 : 1, 1, e->sample_bits, 1, 0, e->stream);
        const float2 *sel_x2 = d_x2 + (half_rot ? kN : 0);
        e->launches += launch_fwd_fft(sel_x2, d_D, e->d_tables, 1, false, e->sm_count, e->stream);
        if ((ce = cudaGetLastError())) break;
        if ((ce = cudaStreamSynchronize(e->stream))) break;
        if (x2 && (ce = cudaMemcpy(x2, sel_x2, kN * sizeof(float2), cudaMemcpyDeviceToHost))) break;
        if (D && (ce = cudaMemcpy(D, d_D, kN * sizeof(float2), cudaMemcpyDeviceToHost))) break;
    } while (0);
    cudaFree(d_pk);
    cudaFree(d_x2);
    cudaFree(d_D);
    cudaFree(d_rot);
    if (ce != cudaSuccess) rc = fail(ACQ_ERR_CUDA, "acq_get_capture_spectrum: %s", cudaGetErrorString(ce));
    return rc;
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
    int kind;
    if (e1b) kind = (ACQ_FORCE_E1B_KERNEL == 2 || (ACQ_FORCE_E1B_KERNEL == 0 && n_tiles <= sm_count / 4)) ? acq::kSearchE1bCluster : acq::kSearchE1b;
    else kind = acq::search_kind_l1(k_noncoh, half_bin);
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
