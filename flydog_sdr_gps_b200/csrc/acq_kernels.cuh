// acq_kernels.cuh -- launch-side declarations shared by acq_kernels.cu and acq_api.cu.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/acq_b200.h"

namespace acq {

// Arguments of the fused correlate + inverse-FFT + peak-search kernel (one "tile" = one
// (capture, satellite, Doppler index); a tile runs k_noncoh inverse FFTs).
struct SearchArgs {
    const float2 *Dp;      // capture spectra, polyphase: [((cap*K + b)*nvar + v)*4 + k2][4096], D[4*k1 + k2]
    const float2 *Ep;      // extended code spectra, polyphase: [(sat*4 + r)][ext_len], E[4*(m - Q) + r]
    const float2 *tables;  // twiddle tables: T2 (kT2Elems), then stage-A bases W16384^{4t+k2} (kBaseElems)
    const int2 *work;      // [n_work] (sat, output slot)
    acq_cell *cells;       // [cap][n_slots][n_dop]
    long long n_tiles;
    int n_work, n_slots, n_dop, dop_lo, half_bin, K, nvar, ext_len, Q;
    // code-Doppler compensation (acq_params.code_doppler): every (block, variant) spectrum exists in n_shift copies,
    // copy i of a block delayed by a further i - smax samples; Doppler index h reads copy smax + s(b, h) of block b,
    // s = round-half-away(b h / cd_div).  n_shift == 1: off.
    int n_shift, smax, cd_div;
    // Small searches: ctas_total > 0 is the number of cell-storing CTAs of the WHOLE search (C/A and E1B launches
    // together); each bumps *ctas_done (zero between searches) after its last cell, and k_pick_small polls it.
    unsigned *ctas_done;
    unsigned ctas_total;
    // Dynamic tile feed of the strided search kernels: a CTA's first tile is its block index, every further one is
    // gridDim.x + atomicAdd(tile_ctr, 1); tile_ctr[2] counts the CTAs that are through with claiming, and the last of
    // them zeroes both words for the next launch.  The C/A and the E1B launch of one search use different pairs
    // (tile_ctr = base + 0 / base + 1).  NULL: static stride.
    unsigned *tile_ctr;
    // k_search_l1_cr claims CHUNKS of consecutive tiles: ck_n16 chunks of 16 tiles, then ck_n4 of 4, then single tiles
    // (filled in by launch_search).
    unsigned ck_n16, ck_n4;
    // 1: wait for the preceding grids of the stream (griddepcontrol.wait).  0: this launch directly follows another
    // search launch of the same search, which has already waited (see launch_search).
    int wait_prior;
    // Aided search (acq_search_aided): dop_center[cap * n_slots + slot] is the raw Doppler centre of that row, which
    // then searches only n_dop = 2 half_width + 1 indices from window_lo(); d of a tile is the index inside the window.
    // NULL: every row searches the engine's whole range dop_lo..dop_hi (n_dop indices).
    const int *dop_center;
    int half_width, dop_hi;
    static constexpr bool kAided = false;
};
// The arguments of an aided search, a type of their own: the search kernels are templates over the argument type and
// read the window only in this instantiation, so the full-range kernels compile to the code they had without the
// feature (k_search_l1_cr sits at 126 registers with its residue loop unrolled: a runtime branch on dop_center moved
// it to 128 and a spill).
struct AidedSearchArgs : SearchArgs {
    static constexpr bool kAided = true;
    AidedSearchArgs() = default;
    explicit AidedSearchArgs(const SearchArgs &a) : SearchArgs(a) {}
};

// s(b, h) of acq_params.code_doppler (same integer arithmetic as the oracle's orc_code_shift)
__host__ __device__ inline int code_shift(int b, int h, int cd_div)
{
    const int a = b * h, m = a < 0 ? -a : a;
    const int s = (2 * m + cd_div) / (2 * cd_div);
    return a < 0 ? -s : s;
}

// First Doppler index of an aided row's window: clamp(center - half_width, dop_lo, dop_hi - 2 half_width), formed
// without overflow for any int32 centre (2 half_width + 1 <= dop_hi - dop_lo + 1, checked by the host).
__host__ __device__ inline int window_lo(int center, int half_width, int dop_lo, int dop_hi)
{
    const int c_lo = dop_lo + half_width, c_hi = dop_hi - half_width;
    const int c = center < c_lo ? c_lo : (center > c_hi ? c_hi : center);
    return c - half_width;
}

// A search launch decomposes its tile index with 32-bit arithmetic; acq_api.cu refuses larger searches.
constexpr long long kMaxTilesPerLaunch = 0x7fffffffLL;

// host-side launchers (all asynchronous on `st`; each returns the number of kernels it launched)
cudaError_t launch_tables_init(const float2 *h_cC, const float *h_hb);
// sample_bits: 1 = the reference's sign-only capture, 2 = sign plane + magnitude plane per block
// n_shift/smax: copies of each output row, copy i delayed by a further i - smax samples (code-Doppler compensation)
int launch_front_end(const uint8_t *packed, float2 *x2, const float2 *rot, int n_blocks, int nvar, int K, int sample_bits,
                     int n_shift, int smax, cudaStream_t st);
int launch_front_end_arg(const uint8_t *packed_host, float2 *x2, const float2 *rot, int nvar, int n_shift, int smax,
                         cudaStream_t st);   // one 1-bit block passed as the kernel's argument (0: launch failed)
int launch_hb1_code(const uint32_t *chips, const int *codelen_boc, float2 *x1, int n_sats, cudaStream_t st);
int launch_hb2(const float2 *x1, float2 *x2, const float2 *rot, int n_rows, int nvar, int K, cudaStream_t st);
// pdl: launch with programmatic stream serialization (the grid may become resident while the previous kernel of
// the stream drains; see pdl_wait() in acq_fft.cuh)
int launch_fwd_fft(const float2 *x2, float2 *out, const float2 *tables, int n_rows, bool polyphase, int sm_count,
                   cudaStream_t st, bool pdl = false);
int launch_build_ext(const float2 *C, float2 *Ep, int n_sats, int Q, int ext_len, int wrap_mode, cudaStream_t st);
int launch_search(const SearchArgs &a, bool e1b, int sm_count, cudaStream_t st, bool pdl = false);
int launch_search_e1b_cluster(const SearchArgs &a, int sm_count, cudaStream_t st, bool pdl = false);
// Doppler indices of the cell rows a best-Doppler pick reads: cell d of row r is index dop_lo + d, or, with
// dop_center (an aided search), window_lo(dop_center[r], half_width, dop_lo, dop_hi) + d.
struct PickDop {
    int dop_lo;
    const int *dop_center;
    int half_width, dop_hi;
};
int launch_best_dop(const acq_cell *cells, const int *slot_sat, acq_record *out, int n_cap, int n_slots, int n_dop,
                    PickDop pd, cudaStream_t st, bool pdl = false);
// best-Doppler pick of a small search: one CTA that polls the search CTAs' counter (see k_pick_small).  host_flag
// (mapped pinned memory, or NULL) selects the polled-host form: `out` is then an acq_record_tagged array in mapped
// memory (tags = epoch), and *host_flag is written only to report a failure (0xffffffff)
int launch_pick_small(const acq_cell *cells, const int *slot_sat, acq_record *out, unsigned *ctas_done, unsigned ctas_total,
                      unsigned *host_flag, unsigned epoch, int n_rows, int n_slots, int n_dop, PickDop pd, cudaStream_t st,
                      bool pdl = false);
// CTAs of a search launch that store cells (what SearchArgs::ctas_total sums over the launches of one search)
enum { kSearchL1 = 0, kSearchE1b = 1, kSearchE1bCluster = 2, kSearchL1Multi = 3, kSearchL1Dr = 4, kSearchL1Mst = 5, kSearchL1Cr = 6 };
int search_kind_l1(int K, int half_bin, long long n_tiles, int sm_count);   // which C/A search kernel (and so which grid) a search uses
// an aided search runs only on the product's search kernels: false where this library would pick another form
bool search_aided_supported(int K, int half_bin, long long tiles_l1, long long tiles_e1b, int sm_count);
constexpr int kPickSmallRowsMax = 256;  // rows k_pick_small stages in shared memory
// A record as k_pick_small hands it to a POLLING host (mapped pinned memory): two 16-byte halves, each carrying the
// search's epoch in its last word.  Each half arrives by one 16-byte store, so a host that sees the epoch in a half has
// the whole half: no system fence and no separate completion word on the kernel's tail.
struct acq_record_tagged {
    int32_t sat, lag, dop;
    uint32_t tag0;
    float peak, noise, snr;
    uint32_t tag1;
};
static_assert(sizeof(acq_record_tagged) == 32, "two 16-byte halves");
int search_grid_ctas(long long n_tiles, int kind, int sm_count);
bool search_claims_tiles(long long n_tiles, int grid);   // tiles claimed from a counter (true) or the static stride
// chunk schedule of k_search_l1_cr (SearchArgs::ck_n16 / ck_n4) and the chunk lengths it was built with
void search_chunks(long long n_tiles, int grid, unsigned *n_big, unsigned *n_mid);
long long search_chunk_count(long long n_tiles, int grid);
void search_chunk_lengths(int *big, int *mid);
// refinement of the records of the most recent search (one CTA per record)
int launch_refine(const float2 *Dp, const float2 *Ep, const acq_record *rec, const int *sat_type, acq_fine *out, int n_rows,
                  int n_slots, int K, int nvar, int half_bin, int ext_len, int Q, int n_shift, int smax, int cd_div,
                  cudaStream_t st);
cudaError_t search_kernels_configure();

}  // namespace acq
