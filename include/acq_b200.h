/*
 * acq_b200.h -- C ABI of the B200-native GNSS acquisition engine.
 *
 * This is the drop-in boundary for the FFT parallel-code-phase search of the reference
 * receiver (FlyDog_SDR_GPS, gps/search.cpp).  The reference has no FFI layer for this path:
 * its boundary is the six free functions of gps/gps.h:140-145 plus the two file-static
 * workers Sample() (gps/search.cpp:382) and Correlate() (gps/search.cpp:453).  Each entry
 * point below names the reference code it replaces.  The host shim that keeps the six
 * SearchXxx symbols and routes them here is include/search_dropin.h (flydog_sdr_gps_b200/csrc/search_dropin.cpp);
 * INTEGRATION.md shows the lines a maintainer changes in the reference tree.
 *
 * Conventions
 *  - plain C: pointers, sizes, POD structs.  No C++/torch/CUDA types cross this boundary
 *    (a CUDA stream is passed as void*).
 *  - every function returns ACQ_OK (0) or a negative acq_status; it never throws or aborts.
 *    acq_last_error() returns a thread-local description of the last failure.
 *  - one engine per GPU; an engine may be driven by one host thread at a time (the reference
 *    search is single-threaded and not re-entrant: gps/search.cpp:51-58,97).
 *  - there is NO CPU fallback: creating an engine without a usable sm_100 device fails.
 */
#ifndef ACQ_B200_H
#define ACQ_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ACQ_ABI_VERSION 3   /* 3: acq_params carries its own size (struct_size first, 64 bytes); 2: code_doppler */

/* Fixed geometry of the reference search (gps/gps.h:60-82, kiwi.config:259). */
#define ACQ_FFT_LEN 16384      /* FFT_LEN */
#define ACQ_NSAMPLES 65536     /* NSAMPLES: 1-bit samples per capture block (4.004 ms at 16.368 MHz) */
#define ACQ_DECIM 4            /* DECIM */
#define ACQ_BLOCK_BYTES 8192   /* 16 SPI packets x 512 B (gps/search.cpp:389-406); sample i = bit i&7 of byte i>>3 */
#define ACQ_LAGS_L1 4092       /* lags scanned for Navstar/QZSS: SAMPLE_RATE/1000 * 1 ms (search.cpp:456,486) */
#define ACQ_LAGS_E1B 16368     /* lags scanned for Galileo E1B: 4 ms code */
#define ACQ_BIN_HZ 249.755859375 /* BIN_SIZE (gps/gps.h:69) */

typedef enum {
    ACQ_OK = 0,
    ACQ_ERR_ARG = -1,         /* bad argument */
    ACQ_ERR_CUDA = -2,        /* CUDA runtime error (text in acq_last_error) */
    ACQ_ERR_NO_DEVICE = -3,   /* no CUDA device / not compute capability 10.x */
    ACQ_ERR_UNSUPPORTED = -4, /* parameter combination not implemented */
    ACQ_ERR_NOMEM = -5
} acq_status;

/* sat_e of the reference (gps/gps.h:98) */
enum { ACQ_NAVSTAR = 0, ACQ_SBAS = 1, ACQ_QZSS = 2, ACQ_E1B = 3 };

/* The leading members of the reference's SATELLITE (gps/gps.h:101-112), same order:
 *   Navstar {prn, T1, T2}     G2 tap pair
 *   QZSS    {prn, G2_delay, G2_init}  (t1 > 10 selects G2-init mode, gps/cacode.h:27-32)
 *   E1B     {prn, 0, 0}       Galileo memory code prn (1..50)
 * "sat" everywhere in this API is the index into the table given to acq_create, exactly
 * like the reference's SATELLITE::sat (gps/search.cpp:186-187). */
typedef struct acq_sat {
    int32_t prn;
    int32_t t1;
    int32_t t2;
    int32_t type;
} acq_sat;

/* How bins past the end of a satellite's doubled code-spectrum row are fetched for negative
 * Doppler.  The compiled reference reads code[sat]+FFT_LEN-dop (gps/search.cpp:471); for dop<0
 * the last |dop| reads fall into the NEXT satellite's row (code[sat+1][0..|dop|-1], zeros after
 * the last satellite).  ACQ_WRAP_REFERENCE reproduces that; ACQ_WRAP_CIRCULAR is the intended
 * C[(k-dop) mod N] (the #else branch, gps/search.cpp:473-477). */
enum { ACQ_WRAP_REFERENCE = 0, ACQ_WRAP_CIRCULAR = 1 };

/* Search parameters.  acq_params_default() fills the values the reference compiles in. */
typedef struct acq_params {
    uint32_t struct_size; /* sizeof(acq_params) of the caller's header, filled by acq_params_default.  acq_create refuses
                             a structure whose size differs from the library's (a caller built against another ABI
                             version would otherwise be read past its end) */
    int32_t dop_lo;     /* first Doppler index, inclusive.  default -20 (gps/search.cpp:465) */
    int32_t dop_hi;     /* last Doppler index, inclusive.   default +20 */
    int32_t half_bin;   /* 0: index = bins of ACQ_BIN_HZ (reference).  1: index = half-bins (extension) */
    int32_t k_noncoh;   /* 1: reference.  K>1: |r|^2 summed over K consecutive blocks (extension) */
    float thr_l1;       /* detection threshold, Navstar/QZSS. default 16 = MIN_SIG / -gsig (search.cpp:70,82-84) */
    float thr_e1b;      /* detection threshold, E1B.          default 16 (search.cpp:549) */
    int32_t wrap_mode;  /* ACQ_WRAP_REFERENCE (default) or ACQ_WRAP_CIRCULAR */
    int32_t sample_bits; /* capture format (this member was "reserved, must be 0"): 0 or 1 = the reference's 1-bit
                            sign-only capture; 2 = 2-bit sign/magnitude (extension, see ACQ_CAPTURE_BLOCK_BYTES) */
    int32_t code_doppler; /* 0 (default): the K-block sum adds block powers at lag n + 16 b.  1: code-Doppler compensation
                             (extension, SURVEY 8(f) rank 4): a carrier offset f stretches the code by f/f_L1, so at
                             Doppler index h block b has advanced a further b*h/385 /DECIM-samples (FS/DECIM/f_L1 =
                             1/385 exactly; h/2 for half-bin indices) and its power is taken at lag
                             n + 16 b + s(b,h), s = that quotient rounded half away from zero.  Recovers the
                             correlation loss of long sums at high Doppler (0.52 chip over 80 ms at 10 kHz); costs
                             (2 max|s| + 1) shifted copies of every capture spectrum (at most ACQ_MAX_CODE_SHIFTS),
                             nothing in the search kernels.  No effect when k_noncoh = 1. */
    int32_t reserved[6];  /* must be 0 */
} acq_params;

#define ACQ_MAX_CODE_SHIFTS 33 /* acq_create fails with ACQ_ERR_UNSUPPORTED when code_doppler needs more shifted copies */

/* Bytes of one 65536-sample capture block in the format `sample_bits` selects.
 *   1 bit : ACQ_BLOCK_BYTES.  Sample i = bit i&7 of byte i>>3 -- the I_sign stream the reference's sampler
 *           delivers (gps/search.cpp:408-411, verilog/gps/gps.v:50,156).
 *   2 bits: 2 * ACQ_BLOCK_BYTES = the sign plane above followed by a MAGNITUDE plane of the same layout
 *           (I_mag of the MAX2769, which the front end is already configured to produce -- dev/gps_fe.cpp:104 --
 *           and the reference's FPGA drops).  A sample is (sign ? -1 : +1) * (mag ? 3 : 1), the MAX2769's
 *           sign/magnitude levels, before the same fs/4 XOR mix.  With an all-zero magnitude plane the results
 *           are bit-identical to the 1-bit format.  No reference counterpart; the oracle carries the same
 *           definition (orc_params.sample_bits). */
#define ACQ_CAPTURE_BLOCK_BYTES(sample_bits) ((sample_bits) == 2 ? 2 * ACQ_BLOCK_BYTES : ACQ_BLOCK_BYTES)

/* One record per (capture, searched satellite): what Correlate() returns (gps/search.cpp:453,495-498)
 * plus the two powers its snr is made of.  24 bytes. */
typedef struct acq_record {
    int32_t sat;  /* table index */
    int32_t lag;  /* max_snr_i: code phase in /DECIM samples, [0, L).  ca_shift = lag*ACQ_DECIM (search.cpp:575) */
    int32_t dop;  /* max_snr_dop: Doppler index (bins, or half-bins when half_bin=1).  lo_shift (search.cpp:574) */
    float peak;   /* max_pwr at that Doppler (search.cpp:488) */
    float noise;  /* ave_pwr at that Doppler (search.cpp:493) */
    float snr;    /* peak/noise = Correlate()'s return value (search.cpp:494,498) */
} acq_record;

/* One cell of the optional per-Doppler table (the values of one iteration of search.cpp:465-496). */
typedef struct acq_cell {
    float peak;
    float noise;
    float snr;
    int32_t lag;
} acq_cell;

/* Refined hand-off values for one record (acq_refine; SURVEY 8(f) rank 4 -- an extension, the reference hands
 * over whole bins and whole /DECIM samples, gps/search.cpp:574-575).  16 bytes. */
typedef struct acq_fine {
    float dop_hz;     /* Doppler in Hz: (bin + three-bin interpolation) * ACQ_BIN_HZ */
    float code_fs;    /* code phase in FS samples: ACQ_DECIM * (lag + early/late interpolation) */
    float peak;       /* |r|^2 at (lag, dop) evaluated directly from the spectra, summed over the K blocks: equals
                         acq_record.peak up to rounding */
    int32_t ca_shift; /* round(code_fs) modulo the code period in FS samples: ChanStart's ca_shift at FS-sample
                         resolution (gps/channel.cpp:925-934) */
} acq_fine;

typedef struct acq_engine acq_engine;

/* Thread-local text of the last error returned on this thread ("" if none). */
const char *acq_last_error(void);
int acq_abi_version(void);

/* Reference defaults: -20..+20 bins, full bins, K=1, thresholds 16, reference wrap, 1-bit captures. */
int acq_params_default(acq_params *p);

/* Replaces SearchInit()'s spectrum build (gps/search.cpp:183-346): generates the C/A (LFSR,
 * gps/cacode.h) and E1B (memory code + BOC(1,1)) replicas, decimates by 4 and transforms them
 * on `device`, and allocates the engine.  sats/n_sats is the caller's satellite table (the
 * reference passes its Sats[]); it is copied.  n_sats is not limited to MAX_SATS=64. */
int acq_create(acq_engine **out, const acq_params *params, const acq_sat *sats, int n_sats, int device);

/* Replaces SearchFree() (gps/search.cpp:354-357). NULL is allowed. */
int acq_destroy(acq_engine *e);

/* Replaces the DSP of Sample() (everything after the SPI reads, gps/search.cpp:408-447) and
 * Correlate() (gps/search.cpp:453-499) for n_sel satellites on n_captures captures in one call.
 *   packed : HOST memory, n_captures * k_noncoh * ACQ_CAPTURE_BLOCK_BYTES(sample_bits) bytes (ACQ_BLOCK_BYTES per
 *            block in the reference's 1-bit format); capture c occupies k_noncoh consecutive blocks.
 *            (Pinned memory avoids a staging copy.  The reference's own search -- ONE 1-bit block -- needs neither:
 *            its 8 KiB travel as the first kernel's launch argument, read from `packed` before the call returns.)
 *   sel    : n_sel table indices to search, or NULL for the whole table (then n_sel is ignored).  Rows of type
 *            ACQ_SBAS carry an all-zero code spectrum, as in the reference (SearchInit builds replicas for Navstar,
 *            QZSS and E1B rows only, gps/search.cpp:244,306): their records are {lag 0, dop 0, snr 0}.
 *   out    : HOST memory, n_captures * n_sel records, record [c*n_sel + s].
 * Synchronous: returns when `out` is filled. */
int acq_search(acq_engine *e, const uint8_t *packed, int n_captures, const int32_t *sel, int n_sel,
               acq_record *out);

/* Same, additionally returning the full per-Doppler table:
 *   grid : HOST memory, n_captures * n_sel * n_dop cells (n_dop = dop_hi-dop_lo+1). */
int acq_search_grid(acq_engine *e, const uint8_t *packed, int n_captures, const int32_t *sel, int n_sel,
                    acq_record *out, acq_cell *grid);

/* Device-resident variant: packed and out are DEVICE pointers on the engine's GPU, work is
 * enqueued on `stream` (a cudaStream_t passed as void*, NULL = the engine's own stream) and the
 * call returns without synchronising.  sel is a HOST array, consumed before returning.
 * packed_dev must be 16-byte aligned (the front end stages the capture with bulk asynchronous copies).
 * Ordering: the engine's scratch (capture spectra, per-Doppler cells, work lists) is shared by all calls.  The engine
 * records an event behind every device-path search and makes whatever touches that scratch next -- a search on
 * another stream, a host-path call, a change of selection or a scratch reallocation -- wait for it, so calls issued
 * from the one driving host thread never overwrite data a running search still reads.  The caller remains
 * responsible for packed_dev / out_dev staying valid until its stream has passed the search. */
int acq_search_device(acq_engine *e, const uint8_t *packed_dev, int n_captures, const int32_t *sel, int n_sel,
                      acq_record *out_dev, void *stream);

/* Aided search: row r = c*n_sel + s (capture c, selected satellite s) searches only the W = 2*half_width+1 Doppler
 * indices [lo_r, lo_r + W - 1], where lo_r = clamp(dop_center[r] - half_width, dop_lo, dop_hi - 2*half_width).
 * Indices are in the engine's units (half-bins when half_bin = 1).  A centre outside the range is clamped, so every
 * row searches a full-width window.  W must not exceed n_dop.  The record is Correlate()'s rule over the window
 * (largest snr, lowest Doppler index on ties, snr > 0), and its dop is the absolute index.
 *   dop_center : HOST, n_captures * n_sel int32 (n_sel = table size when sel is NULL)
 *   grid       : HOST or NULL; n_captures * n_sel * W cells, cell j of row r = Doppler index lo_r + j
 * Synchronous, like acq_search.  acq_refine accepts its records afterwards. */
int acq_search_aided(acq_engine *e, const uint8_t *packed, int n_captures, const int32_t *sel, int n_sel,
                     const int32_t *dop_center, int half_width, acq_record *out, acq_cell *grid);
/* The device-resident form.  Ordering and validity rules are those of acq_search_device; dop_center_dev is a
 * DEVICE array read by the kernels, so it must stay valid until `stream` has passed the search. */
int acq_search_aided_device(acq_engine *e, const uint8_t *packed_dev, int n_captures, const int32_t *sel, int n_sel,
                            const int32_t *dop_center_dev, int half_width, acq_record *out_dev, void *stream);

/* Asynchronous pair over host buffers (the reference yields to other tasks while it computes,
 * gps/search.cpp:479-491): submit enqueues copy-in, search and copy-out on the engine's stream;
 * acq_wait blocks until done, acq_poll returns 1 when done, 0 while running.  The host buffers
 * must stay valid (and `out` unread) until completion. */
int acq_submit(acq_engine *e, const uint8_t *packed, int n_captures, const int32_t *sel, int n_sel,
               acq_record *out);
int acq_poll(acq_engine *e);
int acq_wait(acq_engine *e);

/* Acquisition refinement for the hand-off to tracking.  `rec` (HOST) are the n_captures * n_sel records of the MOST
 * RECENT host-path search on this engine (acq_search, acq_search_grid, acq_search_aided, or acq_submit after acq_wait), in the same
 * order; the capture spectra that search left on the device are reused, so no capture is passed again.  For each
 * record the correlation is evaluated at the five points (dop-1..dop+1 at lag; lag-1..lag+1 at dop), a three-bin
 * Doppler interpolation and an early/late code-phase interpolation are formed, and `out` (HOST, same count) is
 * filled.  Records of undetected satellites are refined like any other (their values are noise).  Returns
 * ACQ_ERR_ARG when there is no completed search, the count differs, or a record does not belong to this engine's
 * table / Doppler range. */
int acq_refine(acq_engine *e, const acq_record *rec, int n_records, acq_fine *out);

/* Detection rule of SearchTask (gps/search.cpp:549,591): snr >= threshold of the sat's type. */
int acq_detected(const acq_engine *e, const acq_record *r);

/* ---- introspection (tests, integration bring-up) ---- */
/* Code spectrum of table entry `sat` as the reference stores it (first copy of code[sat],
 * gps/search.cpp:283): ACQ_FFT_LEN interleaved complex floats to HOST memory. */
int acq_get_code_spectrum(acq_engine *e, int sat, float *out);
/* Front end of one block: packed (HOST, one block in the engine's capture format) -> decimated baseband `x2` (the forward
 * FFT's input, gps/search.cpp:437-445) and spectrum `D` (fwd_buf after search.cpp:447), each
 * ACQ_FFT_LEN interleaved complex floats, either may be NULL.  half_rot=1 selects the
 * half-bin pre-rotated variant. */
int acq_get_capture_spectrum(acq_engine *e, const uint8_t *packed, int half_rot, float *x2, float *D);
/* Satellite table size and parameters the engine was created with. */
int acq_n_sats(const acq_engine *e);
int acq_get_params(const acq_engine *e, acq_params *p);
/* Number of kernels this engine has launched since creation (bench.py's gpu_launches). */
int64_t acq_launch_count(const acq_engine *e);
/* Per-kernel device timing of the most recent search (CUDA events recorded on the launching stream
 * around each kernel when enabled).  acq_get_kernel_ms waits for that search and fills
 *   out[0] = capture front end (unpack + mix + both half-band stages), out[1] = forward FFT,
 *   out[2] = fused correlate + inverse FFT + peak search (all constellations), out[3] = best-Doppler pick (k_pick_small / k_best_dop)
 * in milliseconds; n_out >= 4. */
int acq_set_profiling(acq_engine *e, int enable);
int acq_get_kernel_ms(acq_engine *e, float *out, int n_out);
/* Device ordinal and SM count of the engine's GPU. */
int acq_device_info(const acq_engine *e, int *device, int *sm_count, int *sm_clock_khz);

/* How a search launch of n_tiles tiles (captures x satellites of one family x Doppler indices) would be laid out on a GPU
 * with sm_count SMs: pure host arithmetic, no device needed (tests, bring-up).  e1b: 0 = C/A family, 1 = Galileo E1B.
 *   kernel    : 0 k_search_l1, 1 k_search_e1b, 2 k_search_e1b_cluster, 3 k_search_l1_multi, 6 k_search_l1_cr
 *               (1 also stands for k_search_e1b_multi when k_noncoh > 1)
 *   grid      : CTAs that store cells (clusters count once)
 *   claims    : 1 = the CTAs claim their work from a counter, 0 = static stride blockIdx.x + i * grid
 *   chunk_big / chunk_mid / n_big / n_mid / n_chunks : k_search_l1_cr claims runs of consecutive tiles -- n_big chunks of
 *               chunk_big tiles, then n_mid of chunk_mid, then single tiles; n_chunks in all (other kernels: single
 *               tiles, n_chunks = n_tiles). */
typedef struct acq_launch_plan {
    int32_t kernel, grid, claims, chunk_big, chunk_mid;
    uint32_t n_big, n_mid;
    int64_t n_chunks;
} acq_launch_plan;
int acq_plan_launch(int k_noncoh, int half_bin, int e1b, int64_t n_tiles, int sm_count, acq_launch_plan *out);

/* On-device micro-benchmarks used as roofline denominators (SURVEY 8(d)): fills
 *   out[0] = FP32 FFMA  throughput, TFLOP/s      out[1] = packed FFMA2 throughput, TFLOP/s
 *   out[2] = shared-memory read+write bandwidth, TB/s    out[3] = L2->SM read bandwidth, TB/s
 *   out[4] = SM clock observed during the FFMA run, MHz (cycles/elapsed)
 * n_out >= 5. */
int acq_microbench(int device, double *out, int n_out);

#ifdef __cplusplus
}
#endif
#endif /* ACQ_B200_H */
