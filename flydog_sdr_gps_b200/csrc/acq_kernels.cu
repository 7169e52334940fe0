// acq_kernels.cu -- sm_100a kernels of the acquisition engine.
//
//   K1  k_front_end  : unpack 1-bit (or 2-bit sign/magnitude) capture (TMA-staged), fs/4 XOR mix, both half-band /2 stages
//                      (+ optional half-bin pre-rotation, block delay)              (search.cpp:408-441)
//   K6a k_hb1_code   : C/A / E1B(BOC) replica samples, first half-band /2            (search.cpp:250-275,315-337)
//   K6a' k_hb2       : second half-band /2 of the replica                            (search.cpp:273-275)
//   K2  k_fwd_fft    : 16384-point forward FFT of data or code                       (search.cpp:280,342,447)
//   K6b k_build_ext  : polyphase, margin-extended code-spectrum rows                 (search.cpp:283-284,471)
//   K3-5 k_search_l1 / k_search_e1b : conj(D).C product, 16384-point inverse FFT, |.|^2, non-coherent
//                      sum, max / first-argmax / mean per (capture, sat, Doppler)    (search.cpp:465-494)
//   K5b k_best_dop / search_cta_done : best-snr Doppler per (capture, sat), lowest index on ties (search.cpp:495)
//
// The half-band stages use explicit round-to-nearest mul/add in the reference's summation order
// (no FMA contraction), so the FFT inputs are bit-identical to the reference's x86 build.
#include <cooperative_groups.h>

#include "acq_fft.cuh"
#include "acq_kernels.cuh"

namespace acq {

// half-band taps in the order the reference applies them (search.cpp:141-158):
//   [0] = COEF[0], [1..15] = COEF[2], COEF[4] .. COEF[30], [16] = COEF[15]
__constant__ float c_hb[17];

cudaError_t launch_tables_init(const float2 *h_cC, const float *h_hb)
{
    cudaError_t e = cudaMemcpyToSymbol(c_cC, h_cC, sizeof(float2) * 64);
    if (e != cudaSuccess) return e;
    return cudaMemcpyToSymbol(c_hb, h_hb, sizeof(float) * 17);
}

// ---------------------------------------------------------------------------------------------
// half-band helpers: acc = x[0]*c0; acc += x[j]*c_j (j = 2,4..30); acc += x[15]*c15
// ---------------------------------------------------------------------------------------------
struct HbAcc {
    float re, im;
    __device__ __forceinline__ void first(float xr, float xi, float c)
    {
        re = __fmul_rn(xr, c);
        im = __fmul_rn(xi, c);
    }
    __device__ __forceinline__ void add(float xr, float xi, float c)
    {
        re = __fadd_rn(re, __fmul_rn(xr, c));
        im = __fadd_rn(im, __fmul_rn(xi, c));
    }
};

// K1.  Fused capture front end: unpack + fs/4 XOR mix + both half-band /2 stages, one launch.
// A CTA produces kFeOut = 1024 consecutive samples of x2 for one 65536-sample block.  It needs x1[2 o0 .. 2 o0 + 2077],
// i.e. capture bits 4 o0 .. 4 o0 + 4185 = 524 bytes starting at byte 512*chunk: the packed bytes are staged
// into shared memory by ONE bulk asynchronous copy (TMA, cp.async.bulk + mbarrier complete_tx; SASS UBLKCP),
// x1 is formed in shared memory (never written to HBM), then x2.
// Sample i of the block is bit i&7 of byte i>>3 (search.cpp:408-411); LO phase is i&3 (lo_rate == 1,
// search.cpp:386,422-423); I = bit ^ {1,1,0,0}[i&3], Q = bit ^ {1,0,0,1}[i&3]; value = bit ? -1 : +1
// (search.cpp:62-66,172-175).  Past the end of the block both stages see zeros (search.cpp:145).
// Second stage as k_hb2 (optional half-bin variant, block delay for non-coherent sums).
// Chunk size: 256 samples of x2 per CTA (64 CTAs per block).  Measured on one cold-start search with the trace variant
// (round 2, after the first stage went bit-parallel): the front end's last CTA exits at 3.9 us with 1024-sample
// chunks, 2.4 us with 512, 1.6 us with 256, and the whole search ends 3 us earlier; the 30-sample window overlap costs
// 6 % more first-stage work, nothing against a step of a batched search (front end < 1 % there).
#ifndef ACQ_FE_OUT
#define ACQ_FE_OUT 256
#endif
constexpr int kFeOut = ACQ_FE_OUT;             // x2 samples per CTA (a power of two, 256..1024)
constexpr int kFeX1 = 2 * kFeOut + 30;         // x1 samples needed (2078 for 1024)
constexpr int kFeChunkBytes = kFeOut / 2;      // capture bytes that belong to the chunk (4 bits per x2 sample)
constexpr int kFeBytes = (kFeChunkBytes + 12 + 15) / 16 * 16 + 16;  // staged bytes: chunk + 88 bits of look-ahead, 16-byte units

//
// MAG (2-bit sign/magnitude capture, acq_params.sample_bits = 2 -- the MAX2769's native output, of which the
// reference's FPGA keeps the sign only, verilog/gps/gps.v:50): a block is the sign plane (the 1-bit format above)
// followed by a magnitude plane of the same layout; the mixed sample is (bit ? -1 : +1) * (mag ? 3 : 1).  Both
// planes are staged by bulk copies on the same mbarrier.  The products with the taps stay exact roundings of
// (+-1 | +-3) * c in the reference's summation order.
// Code-Doppler compensation (n_shift > 1): every output row is written n_shift times, copy i delayed by a further
// i - smax samples (row layout [block][variant][copy][16384]); the search kernels pick the copy per (block, Doppler).
// A single 1-bit block can also ride in the launch itself (k_front_end_arg below: the capture is a kernel argument, so the
// host path needs no copy node before the first kernel); the body is shared, only the staging of the packed bytes differs.
struct FeBlockArg {
    uint32_t w[ACQ_BLOCK_BYTES / 4];
};
template <bool MAG, bool FROM_ARG>
__device__ __forceinline__ void front_end_body(const uint8_t *__restrict__ packed, const FeBlockArg *__restrict__ arg,
                                               float2 *__restrict__ x2, const float2 *__restrict__ rot, int nvar, int K,
                                               int row0, int n_shift, int smax)
{
    __shared__ __align__(16) uint8_t sbits[kFeBytes + 16];
    __shared__ __align__(16) uint8_t mbits[MAG ? kFeBytes + 16 : 16];
    __shared__ __align__(8) unsigned long long bar;
    __shared__ float2 x1s[kFeX1 + 2];
    const int t = threadIdx.x;
    ACQ_TRACE_STAMP(kTrFrontEnd, 0);
    pdl_launch_dependents();
    const int chunk = blockIdx.x;                      // kN / kFeOut chunks per block
    const int avail = ACQ_BLOCK_BYTES - kFeChunkBytes * chunk;  // bytes of this block from the chunk start
    const int nbytes = avail < kFeBytes ? avail : kFeBytes;     // the last chunk(s): never read past the block
    if (FROM_ARG) {
        // the chunk's bytes straight from the argument (constant bank): word i of the staged window = word i of the chunk
        static_assert(kFeChunkBytes % 4 == 0 && kFeBytes % 4 == 0 && (kFeBytes + 16) % 4 == 0, "word-wise staging");
        uint32_t *sw = reinterpret_cast<uint32_t *>(sbits);
        const int w0 = (kFeChunkBytes / 4) * chunk;
        for (int i = t; i < (kFeBytes + 16) / 4; i += 256) sw[i] = (4 * i < nbytes) ? arg->w[w0 + i] : 0u;
        __syncthreads();
    } else {
        const uint8_t *pk = packed + (size_t)blockIdx.y * (MAG ? 2 : 1) * ACQ_BLOCK_BYTES + kFeChunkBytes * chunk;
        const uint32_t bar_a = (uint32_t)__cvta_generic_to_shared(&bar);
        const uint32_t dst_a = (uint32_t)__cvta_generic_to_shared(sbits);
        if (t == 0) {
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar_a) : "memory");
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        for (int i = nbytes + t; i < kFeBytes + 16; i += 256) {  // zero tail (samples past the block)
            sbits[i] = 0;
            if (MAG) mbits[i] = 0;
        }
        __syncthreads();
        if (t == 0) {
            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar_a), "r"((MAG ? 2 : 1) * nbytes) : "memory");
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst_a),
                         "l"(pk), "r"(nbytes), "r"(bar_a)
                         : "memory");
            if (MAG)
                asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                                 (uint32_t)__cvta_generic_to_shared(mbits)),
                             "l"(pk + ACQ_BLOCK_BYTES), "r"(nbytes), "r"(bar_a)
                             : "memory");
        }
        {   // every thread waits for the bytes to land (phase 0)
            mbar_wait(bar_a, 0);
        }
    }
    // ---- first half-band stage into shared memory: x1s[m] = x1[2*o0 + m]
    const int i_base = 4 * kFeOut * chunk;  // first capture sample of this chunk (= bit 0 of sbits)
    for (int m = t; m < kFeX1; m += 256) {
        const int r0 = 2 * m;  // chunk-relative sample index of the first tap
        if (!MAG && i_base + r0 + 30 < ACQ_NSAMPLES) {
            // Sign-only samples, window inside the block (all but the last 15 outputs of a block): the 31 bits under the
            // taps come from two 32-bit shared loads and a funnel shift; XORing them with the fs/4 LO patterns of the
            // window's phase (I: {1,1,0,0}, Q: {1,0,0,1} per sample, search.cpp:383-384; the window starts at phase 0
            // or 2) leaves each tap's sign in one bit.  A tap product (+-1) * c is exactly +-c, so it is the tap with
            // its sign bit flipped -- the same value __fmul_rn gives -- added in the reference's order with __fadd_rn.
            const uint32_t *w32 = reinterpret_cast<const uint32_t *>(sbits);
            const uint32_t win = __funnelshift_r(w32[r0 >> 5], w32[(r0 >> 5) + 1], r0 & 31);
            const bool ph2 = (r0 & 2) != 0;
            const uint32_t sI = win ^ (ph2 ? 0xCCCCCCCCu : 0x33333333u), sQ = win ^ (ph2 ? 0x66666666u : 0x99999999u);
            auto term = [](uint32_t sgn, int j, float c) {
                return __int_as_float(__float_as_int(c) ^ (int)((sgn << (31 - j)) & 0x80000000u));
            };
            float re = term(sI, 0, c_hb[0]), im = term(sQ, 0, c_hb[0]);
#pragma unroll
            for (int j = 2; j <= 30; j += 2) {
                re = __fadd_rn(re, term(sI, j, c_hb[j / 2]));
                im = __fadd_rn(im, term(sQ, j, c_hb[j / 2]));
            }
            re = __fadd_rn(re, term(sI, 15, c_hb[16]));
            im = __fadd_rn(im, term(sQ, 15, c_hb[16]));
            x1s[m] = (2 * kFeOut * chunk + m < 32768) ? make_float2(re, im) : make_float2(0.0f, 0.0f);
            continue;
        }
        unsigned long long win = 0;
#pragma unroll
        for (int k = 0; k < 5; k++) win |= (unsigned long long)sbits[(r0 >> 3) + k] << (8 * k);
        win >>= (r0 & 7);
        unsigned long long mwin = 0;
        if (MAG) {
#pragma unroll
            for (int k = 0; k < 5; k++) mwin |= (unsigned long long)mbits[(r0 >> 3) + k] << (8 * k);
            mwin >>= (r0 & 7);
        }
        auto sample = [&](int j, float &xr, float &xi) {
            const int i = i_base + r0 + j;
            if (i < ACQ_NSAMPLES) {
                const unsigned bit = (unsigned)(win >> j) & 1u;
                const unsigned ph = i & 3;
                const unsigned lsin = (ph < 2) ? 1u : 0u;             // {1,1,0,0}
                const unsigned lcos = (ph == 0 || ph == 3) ? 1u : 0u; // {1,0,0,1}
                const float w = (MAG && ((unsigned)(mwin >> j) & 1u)) ? 3.0f : 1.0f;
                xr = (bit ^ lsin) ? -w : w;
                xi = (bit ^ lcos) ? -w : w;
            } else {  // zero padding past the end of the block (search.cpp:145)
                xr = 0.0f;
                xi = 0.0f;
            }
        };
        HbAcc acc;
        float xr, xi;
        sample(0, xr, xi);
        acc.first(xr, xi, c_hb[0]);
#pragma unroll
        for (int j = 2; j <= 30; j += 2) {
            sample(j, xr, xi);
            acc.add(xr, xi, c_hb[j / 2]);
        }
        sample(15, xr, xi);
        acc.add(xr, xi, c_hb[16]);
        // x1 has 32768 samples; the second stage pads with zeros beyond (search.cpp:145)
        x1s[m] = (2 * kFeOut * chunk + m < 32768) ? make_float2(acc.re, acc.im) : make_float2(0.0f, 0.0f);
    }
    __syncthreads();
    // ---- second half-band stage: x2[o0 + oo] from x1s[2*oo + j]
    float2 *out = x2 + (size_t)blockIdx.y * nvar * n_shift * kN;
    const int delay = 16 * (int)((row0 + blockIdx.y) % K) - smax;
    for (int oo = t; oo < kFeOut; oo += 256) {
        const float2 *in = x1s + 2 * oo;
        HbAcc acc;
        float2 v = in[0];
        acc.first(v.x, v.y, c_hb[0]);
#pragma unroll
        for (int j = 2; j <= 30; j += 2) {
            v = in[j];
            acc.add(v.x, v.y, c_hb[j / 2]);
        }
        v = in[15];
        acc.add(v.x, v.y, c_hb[16]);
        const int o = kFeOut * chunk + oo;
        const float2 y = make_float2(acc.re, acc.im);
        for (int i = 0; i < n_shift; i++) out[(size_t)i * kN + ((o + delay + i) & (kN - 1))] = y;
        if (nvar == 2) {
            const float2 w = rot[o];
            const float2 yh = make_float2(__fsub_rn(__fmul_rn(acc.re, w.x), __fmul_rn(acc.im, w.y)),
                                          __fadd_rn(__fmul_rn(acc.re, w.y), __fmul_rn(acc.im, w.x)));
            for (int i = 0; i < n_shift; i++) out[(size_t)(n_shift + i) * kN + ((o + delay + i) & (kN - 1))] = yh;
        }
    }
    ACQ_TRACE_STAMP(kTrFrontEnd, 2);
}

template <bool MAG>
__global__ void __launch_bounds__(256) k_front_end(const uint8_t *__restrict__ packed, float2 *__restrict__ x2,
                                                   const float2 *__restrict__ rot, int nvar, int K, int row0,
                                                   int n_shift, int smax)
{
    front_end_body<MAG, false>(packed, nullptr, x2, rot, nvar, K, row0, n_shift, smax);
}

// One 1-bit block handed over as a kernel argument (8 KiB of the 32 KiB a launch may carry): a single-capture search
// through acq_search then starts with this kernel -- no staging memcpy, no copy node, no copy-engine-to-SM hand-over.
__global__ void __launch_bounds__(256) k_front_end_arg(const __grid_constant__ FeBlockArg block, float2 *__restrict__ x2,
                                                       const float2 *__restrict__ rot, int nvar, int n_shift, int smax)
{
    front_end_body<false, true>(nullptr, &block, x2, rot, nvar, 1, 0, n_shift, smax);
}

// K6a.  Replica: sample i carries chip (i>>4) mod codelen (ca_rate = 1/16 exactly, search.cpp:205,254-258),
// E1B XORs the BOC(1,1) sub-carrier (i&15) >= 8 (search.cpp:317-318).  Imaginary part is zero (search.cpp:266).
__global__ void __launch_bounds__(256) k_hb1_code(const uint32_t *__restrict__ chips,
                                                  const int *__restrict__ codelen_boc, float2 *__restrict__ x1)
{
    const int o = blockIdx.x * 256 + threadIdx.x;
    const int sat = blockIdx.y;
    const uint32_t *cw = chips + (size_t)sat * 128;
    const int codelen = codelen_boc[2 * sat];
    const int boc = codelen_boc[2 * sat + 1];
    const int i0 = 2 * o;
    auto sample = [&](int j) -> float {
        const int i = i0 + j;
        if (i >= ACQ_NSAMPLES || codelen == 0) return 0.0f;  // codelen 0: a row the reference builds no replica for (SBAS)
        const int ci = (i >> 4) % codelen;
        unsigned c = (cw[ci >> 5] >> (ci & 31)) & 1u;
        if (boc) c ^= ((i & 15) >= 8) ? 1u : 0u;
        return c ? -1.0f : 1.0f;
    };
    float acc = __fmul_rn(sample(0), c_hb[0]);
#pragma unroll
    for (int j = 2; j <= 30; j += 2) acc = __fadd_rn(acc, __fmul_rn(sample(j), c_hb[j / 2]));
    acc = __fadd_rn(acc, __fmul_rn(sample(15), c_hb[16]));
    x1[(size_t)sat * 32768 + o] = make_float2(acc, 0.0f);
}

// K1b.  Second half-band stage, 32768 -> 16384 per row.  With nvar == 2 also writes the half-bin
// variant x2[n] * exp(-j*pi*n/N) (rot[] is computed on the host in double precision).
// x2 layout: [row][v][16384].
// Non-coherent mode (K > 1): block b = row % K of a capture is stored circularly delayed by 16*b samples,
// x2'[(n + 16 b) mod N] = x2[n], which makes its correlation r'_b[n] = r_b[(n + 16 b) mod N]: the
// 16-lag-per-block code advance (65536 = 4 x 16368 + 64 samples) is removed before the FFT, so the
// search kernel can add block powers lag by lag in registers.
__global__ void __launch_bounds__(256) k_hb2(const float2 *__restrict__ x1, float2 *__restrict__ x2,
                                             const float2 *__restrict__ rot, int nvar, int K, int row0)
{
    const int o = blockIdx.x * 256 + threadIdx.x;
    const float2 *in = x1 + (size_t)blockIdx.y * 32768;
    const int i0 = 2 * o;
    auto sample = [&](int j) -> float2 {
        const int i = i0 + j;
        return (i < 32768) ? in[i] : make_float2(0.0f, 0.0f);
    };
    HbAcc acc;
    float2 v = sample(0);
    acc.first(v.x, v.y, c_hb[0]);
#pragma unroll
    for (int j = 2; j <= 30; j += 2) {
        v = sample(j);
        acc.add(v.x, v.y, c_hb[j / 2]);
    }
    v = sample(15);
    acc.add(v.x, v.y, c_hb[16]);
    float2 *out = x2 + (size_t)blockIdx.y * nvar * kN;
    const int oo = (o + 16 * (int)((row0 + blockIdx.y) % K)) & (kN - 1);
    out[oo] = make_float2(acc.re, acc.im);
    if (nvar == 2) {
        const float2 w = rot[o];
        out[kN + oo] = make_float2(__fsub_rn(__fmul_rn(acc.re, w.x), __fmul_rn(acc.im, w.y)),
                                  __fadd_rn(__fmul_rn(acc.re, w.y), __fmul_rn(acc.im, w.x)));
    }
}

// ---------------------------------------------------------------------------------------------
// K2.  Forward 16384-point FFT of one row per CTA:  Y = conj( IFFT( conj(x) ) ).
// The four sub-FFT outputs of a lag are produced by the same thread, so the radix-4 combine over
// k2 uses a thread-private shared scratch Z (three residues parked, the fourth in registers).
// POLY: write Y in the polyphase layout the search kernel reads ([k2][k1] = Y[4*k1 + k2]).
// ---------------------------------------------------------------------------------------------
constexpr size_t kZBytes = sizeof(float2) * 3 * 16 * 256;

__device__ __forceinline__ void load_t2(const FftSmem3 &s, const float2 *__restrict__ tables, int t)
{
    const float4 *src = reinterpret_cast<const float4 *>(tables);
    float4 *dst = reinterpret_cast<float4 *>(s.T2);
    for (int i = t; i < kT2Elems / 2; i += 256) dst[i] = __ldg(src + i);
    __syncthreads();
}

template <bool POLY>
__global__ void __launch_bounds__(256, 1) k_fwd_fft(const float2 *__restrict__ x2, float2 *__restrict__ out,
                                                    const float2 *__restrict__ tables, int n_rows)
{
    extern __shared__ __align__(1024) unsigned char smem[];
    const FftSmem3 s = fft_smem3_carve(smem);
    float2 *Z = reinterpret_cast<float2 *>(smem + fft_smem3_bytes());
    const int t = threadIdx.x;
    ACQ_TRACE_STAMP(kTrFwdFft, 0);
    pdl_trigger_fft();
    load_t2(s, tables, t);
    const float2 *base = tables + kT2Elems + t;
    int buf = 0;
    pdl_wait();
    ACQ_TRACE_STAMP(kTrFwdFft, 1);
    for (int row = blockIdx.x; row < n_rows; row += gridDim.x) {
        const float2 *in = x2 + (size_t)row * kN;
        float2 *o = out + (size_t)row * kN;
        float2 x[16];
#pragma unroll 1
        for (int k2 = 0; k2 < 4; k2++) {
#pragma unroll
            for (int a = 0; a < 16; a++) {
                const float2 v = in[1024 * a + 4 * t + k2];
                x[a] = make_float2(v.x, -v.y);
            }
            subfft4096_inv3(x, k2, __ldg(base + k2 * 256), buf, s, t);
            buf ^= 1;
            if (k2 < 3) {
#pragma unroll
                for (int n2 = 0; n2 < 16; n2++) {
                    const float2 z = (k2 == 0) ? x[r16(n2)] : cmul(x[r16(n2)], c_cC[k2][n2]);
                    Z[(k2 * 16 + n2) * 256 + t] = z;
                }
            }
        }
#pragma unroll
        for (int n2 = 0; n2 < 16; n2++) {
            float2 z0 = Z[(0 * 16 + n2) * 256 + t];
            float2 z1 = Z[(1 * 16 + n2) * 256 + t];
            float2 z2 = Z[(2 * 16 + n2) * 256 + t];
            float2 z3 = cmul(x[r16(n2)], c_cC[3][n2]);
            radix4_inv(z0, z1, z2, z3);  // z_m = sum_k2 z_k2 * j^{k2*m}
            const float2 zz[4] = {z0, z1, z2, z3};
#pragma unroll
            for (int m = 0; m < 4; m++) {
                const int n = lag_of3(t, n2) + 4096 * m;
                const float2 y = make_float2(zz[m].x, -zz[m].y);
                if (POLY) o[(n & 3) * 4096 + (n >> 2)] = y;
                else o[n] = y;
            }
        }
        // Z is thread-private and the S1/S2 hazards are covered inside subfft4096_inv3: no barrier needed.
    }
}

// K2, cluster form for a handful of rows (single-capture searches, where one CTA per row leaves the GPU idle and
// the forward FFT is a serial 4-sub-FFT chain): a cluster of four CTAs per row, CTA k2 runs one sub-FFT, the
// radix-4 combine reads the other CTAs' outputs through DSMEM (slices of n', as in k_search_e1b_cluster).
template <bool POLY>
__global__ void __cluster_dims__(4, 1, 1) __launch_bounds__(256, 1)
    k_fwd_fft_cluster(const float2 *__restrict__ x2, float2 *__restrict__ out, const float2 *__restrict__ tables,
                      int n_rows)
{
    namespace cg = cooperative_groups;
    cg::cluster_group cluster = cg::this_cluster();
    extern __shared__ __align__(1024) unsigned char smem[];
    const FftSmem3 s = fft_smem3_carve(smem);
    float2 *Y = reinterpret_cast<float2 *>(smem + fft_smem3_bytes());  // [2][16][256]
    const int t = threadIdx.x;
    const int rank = (int)cluster.block_rank();
    ACQ_TRACE_STAMP(kTrFwdFft, 0);
    pdl_trigger_fft();
    load_t2(s, tables, t);
    const float2 bw = __ldg(tables + kT2Elems + rank * 256 + t);
    const float2 *Yr[4];
#pragma unroll
    for (int k = 0; k < 4; k++) Yr[k] = cluster.map_shared_rank(Y, k);
    const int n_clusters = gridDim.x >> 2;
    int buf = 0, yb = 0;
    pdl_wait();
    ACQ_TRACE_STAMP(kTrFwdFft, 1);
    for (int row = blockIdx.x >> 2; row < n_rows; row += n_clusters) {
        const float2 *in = x2 + (size_t)row * kN;
        float2 *o = out + (size_t)row * kN;
        float2 x[16];
#pragma unroll
        for (int a = 0; a < 16; a++) {
            const float2 v = in[1024 * a + 4 * t + rank];
            x[a] = make_float2(v.x, -v.y);
        }
#ifdef ACQ_TRACE
        if (x[15].x == 1.2345e38f) out[0] = x[15];   // (never true) the stamp below waits for the loads
        if (t == 0) { unsigned long long tm; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(tm)); g_trace[kTrFwdFft][64 + blockIdx.x][3] = tm; }
#endif
        subfft4096_inv3(x, rank, bw, buf, s, t);
#ifdef ACQ_TRACE
        if (t == 0) { unsigned long long tm; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(tm)); g_trace[kTrFwdFft][128 + blockIdx.x][3] = tm; }
#endif
        buf ^= 1;
        float2 *Yw = Y + yb * kSub;
#pragma unroll
        for (int n2 = 0; n2 < 16; n2++) Yw[n2 * 256 + t] = (rank == 0) ? x[r16(n2)] : cmul(x[r16(n2)], c_cC[rank][n2]);
        cluster.sync();
#ifdef ACQ_TRACE
        if (t == 0) { unsigned long long tm; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(tm)); g_trace[kTrFwdFft][192 + blockIdx.x][3] = tm; }
#endif
        // all sixteen DSMEM loads first (twelve of them remote): behind the stores of an earlier slice -- which the
        // compiler must assume could alias a mapped shared-memory pointer -- they would be four dependent round trips
        // (trace variant: 1.9-2.2 us for this loop before, of a 5 us kernel)
        float2 zin[4][4];
#pragma unroll
        for (int i = 0; i < 4; i++) {
            const int oidx = yb * kSub + (4 * rank + i) * 256 + t;
#pragma unroll
            for (int k = 0; k < 4; k++) zin[i][k] = Yr[k][oidx];
        }
        // this CTA is through with the other CTAs' shared memory: arrive now (release orders the loads above before it),
        // wait after the stores -- the barrier's latency hides behind the combine instead of ending the kernel
        cluster.barrier_arrive();
#pragma unroll
        for (int i = 0; i < 4; i++) {
            const int n2 = 4 * rank + i;
            float2 z0 = zin[i][0], z1 = zin[i][1], z2 = zin[i][2], z3 = zin[i][3];
            radix4_inv(z0, z1, z2, z3);
            const float2 zz[4] = {z0, z1, z2, z3};
#pragma unroll
            for (int m = 0; m < 4; m++) {
                const int n = lag_of3(t, n2) + 4096 * m;
                const float2 y = make_float2(zz[m].x, -zz[m].y);
                if (POLY) o[(n & 3) * 4096 + (n >> 2)] = y;
                else o[n] = y;
            }
        }
#ifdef ACQ_TRACE
        if (t == 0) { unsigned long long tm; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(tm)); g_trace[kTrFwdFft][256 + blockIdx.x][3] = tm; }
#endif
        yb ^= 1;  // Y is double buffered: a buffer is rewritten two rows later, after the next cluster barrier
        cluster.barrier_wait();  // no CTA may go on (or exit) while another still reads its shared memory
    }
    ACQ_TRACE_STAMP(kTrFwdFft, 2);
}

// ---------------------------------------------------------------------------------------------
// K6b.  Extended polyphase rows of the code spectra:
//   Ep[(sat*4 + r)][mm] = E_sat[4*(mm - Q) + r],   E_sat[j] = C_sat[j mod N]          for j <  N
//                                                            = C_{sat+1}[j - N] or 0   for j >= N, reference wrap
//                                                            = C_sat[j - N]            for j >= N, circular wrap
// so that the product for Doppler bin `dop` reads E_sat[k - dop] with no modulo (the reference gets
// the same effect from its doubled rows, search.cpp:54,283-284,471).
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_build_ext(const float2 *__restrict__ C, float2 *__restrict__ Ep, int n_sats,
                                                   int Q, int ext_len, int wrap_mode)
{
    const int mm = blockIdx.x * 256 + threadIdx.x;
    if (mm >= ext_len) return;
    const int sat = blockIdx.y >> 2, r = blockIdx.y & 3;
    const int j = 4 * (mm - Q) + r;
    float2 v;
    if (j < 0) v = C[(size_t)sat * kN + j + kN];
    else if (j < kN) v = C[(size_t)sat * kN + j];
    else if (wrap_mode == ACQ_WRAP_CIRCULAR) v = C[(size_t)sat * kN + j - kN];
    else v = (sat + 1 < n_sats) ? C[(size_t)(sat + 1) * kN + j - kN] : make_float2(0.0f, 0.0f);
    Ep[(size_t)blockIdx.y * ext_len + mm] = v;
}

// ---------------------------------------------------------------------------------------------
// K3-5.  The search kernels.  Persistent CTAs stride over tiles = (capture, satellite, Doppler index); a tile
// runs K inverse FFTs of 16384 points as four 4096-point sub-FFTs (one per input residue k2).
//   k_search_l1<MULTI> : Navstar / QZSS / SBAS, lags 0..4091 -- only m = 0 of the radix-4 combine is formed,
//                        so the combine is an accumulation in registers.  Two 256-thread CTAs per SM.
//                        MULTI (k_noncoh > 1): block powers summed in registers,
//                        P[n] += |r_b[(n + 16 b) mod N]|^2; the 16-lag-per-block code advance is removed
//                        in the front end by delaying block b (see k_hb2).
//   k_search_e1b       : Galileo E1B, lags 0..16367 -- three residues are parked in thread-private TENSOR MEMORY
//                        (tcgen05.st / tcgen05.ld) and all four m are formed.  Two CTAs per SM.
// ---------------------------------------------------------------------------------------------
struct Peak {
    float p;
    int n;
    float sum;
};

__device__ __forceinline__ void peak_merge(Peak &a, float p, int n, float sum)
{
    if (p > a.p || (p == a.p && n < a.n)) {  // first (lowest) index wins ties, search.cpp:488
        a.p = p;
        a.n = n;
    }
    a.sum += sum;
}

__device__ __forceinline__ Peak block_reduce_peak(Peak v, float *red_f, int *red_i, int t)
{
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        const float p = __shfl_xor_sync(0xffffffffu, v.p, off);
        const int n = __shfl_xor_sync(0xffffffffu, v.n, off);
        const float s = __shfl_xor_sync(0xffffffffu, v.sum, off);
        peak_merge(v, p, n, s);
    }
    const int w = t >> 5;
    if ((t & 31) == 0) {
        red_f[w] = v.p;
        red_f[8 + w] = v.sum;
        red_i[w] = v.n;
    }
    __syncthreads();
    if (t == 0) {
        v.p = red_f[0];
        v.n = red_i[0];
        v.sum = red_f[8];
#pragma unroll
        for (int k = 1; k < 8; k++) peak_merge(v, red_f[k], red_i[k], red_f[8 + k]);
    }
    return v;  // valid in thread 0
}

struct TileIdx {
    int sat, slot, cap, d, dop, v, wi;
    __device__ __forceinline__ TileIdx() {}
    // The host keeps a launch below 2^31 tiles (launch_search), so the decomposition runs on 32-bit unsigned
    // divisions: every warp pays it once per tile, and a K = 1 tile is only four sub-FFTs long.
    template <class PA>
    __device__ __forceinline__ TileIdx(const PA &p, long long tile)
    {
        const unsigned tl = (unsigned)tile, nd = (unsigned)p.n_dop, nw = (unsigned)p.n_work;
        const unsigned cw = tl / nd;
        d = (int)(tl - cw * nd);
        cap = (int)(cw / nw);
        wi = (int)(cw - (unsigned)cap * nw);
        const int2 wk = p.work[wi];
        sat = wk.x;
        slot = wk.y;
        set_dop(p);
    }
    // the tile `stride` further on, stride given as mixed-radix digits (sd, sw, sc) over (n_dop, n_work): no division
    template <class PA>
    __device__ __forceinline__ void step(const PA &p, int sd, int sw, int sc)
    {
        d += sd;
        int carry = d >= p.n_dop;
        if (carry) d -= p.n_dop;
        wi += sw + carry;
        carry = wi >= p.n_work;
        if (carry) wi -= p.n_work;
        cap += sc + carry;
        const int2 wk = p.work[wi];
        sat = wk.x;
        slot = wk.y;
        set_dop(p);
    }
    // Doppler index h of the tile: dop_lo + d, or in an aided search (AidedSearchArgs) d steps into its row's window.  The
    // claiming kernels form a tile's indices in the one thread that publishes them, so the centre's load stays there.
    template <class PA>
    __device__ __forceinline__ void set_dop(const PA &p)
    {
        int h;
        if constexpr (PA::kAided) h = window_lo(__ldg(p.dop_center + cap * p.n_slots + slot), p.half_width, p.dop_lo, p.dop_hi) + d;
        else h = p.dop_lo + d;
        v = p.half_bin ? (h & 1) : 0;
        dop = p.half_bin ? ((h - v) >> 1) : h;
    }
};

// Dynamic tile feed of the strided search kernels (k_search_l1, k_search_l1_multi, k_search_e1b, k_search_e1b_multi).
// Two CTAs share an SM, and the SM does not share itself evenly: with a static stride the CTA that became resident first
// ran its tiles 1.4-1.9x faster than its neighbour (%globaltimer stamps, trace variant: K = 20 C/A search, CTAs 0..147
// done at 2.59 ms, CTAs 148..295 at 3.63 ms; E1B search 123 us against 171-179 us), and the late half then finished
// alone on its SM at 1.3x, not 2x, the shared rate.  So a CTA takes tile blockIdx.x first and claims every further one
// from a counter: thread 0 draws the claim during the tile's first sub-FFT (the atomic's latency is off every chain),
// publishes the next tile's indices in shared memory after the barrier of the second-to-last sub-FFT, stages that tile's
// first operands after the last barrier, and every thread picks the indices up behind that barrier.  Every CTA counts
// itself out after its last claim, and the last one out resets both counters (claims_done).
// Cells do not depend on which CTA computes them: results are bit-identical to the static stride.
// `cur`: the tile the CTA is running.  tile_ctr == NULL: the static stride (successor cur + gridDim.x) -- searches of only
// a few rounds, see search_claims_tiles().
// (Tried against the greedy tail and dropped: the late-resident CTA of each SM -- block index in the upper half of the
// grid -- stops claiming once no more than one tile per SM is left, so that the last tiles run one per SM.  Slower
// everywhere: 32 PRNs x 41 bins 80.1 us against 78.8 us through acq_search, the 82-PRN search 167.9 against 164.4 us.)
constexpr unsigned kNoTile = 0xffffffffu;
__device__ __forceinline__ unsigned claim_tile(const SearchArgs &p, unsigned cur)
{
    if (!p.tile_ctr) return cur + gridDim.x;
    return gridDim.x + atomicAdd(p.tile_ctr, 1u);
}
// End of a claiming CTA (after its last claim): the last one out puts both counters back to zero for the next launch.
__device__ __forceinline__ void claims_done(const SearchArgs &p, int t)
{
    if (p.tile_ctr && t == 0 && atomicAdd(p.tile_ctr + 2, 1u) == gridDim.x - 1) {
        *(volatile unsigned *)p.tile_ctr = 0u;
        *(volatile unsigned *)(p.tile_ctr + 2) = 0u;
    }
}
template <class PA>
__device__ __forceinline__ void publish_tile(int *feed, const PA &p, unsigned nxt)   // one thread
{
    if (nxt < (unsigned)p.n_tiles) {
        const TileIdx tn(p, nxt);
        feed[1] = tn.sat, feed[2] = tn.slot, feed[3] = tn.cap, feed[4] = tn.d, feed[5] = tn.dop, feed[6] = tn.v, feed[7] = tn.wi;
        feed[0] = 1;
    } else {
        feed[0] = 0;
    }
}
__device__ __forceinline__ bool next_tile(const int *feed, TileIdx &ti)
{
    if (!feed[0]) return false;
    ti.sat = feed[1], ti.slot = feed[2], ti.cap = feed[3], ti.d = feed[4], ti.dop = feed[5], ti.v = feed[6], ti.wi = feed[7];
    return true;
}

// Row of the capture-spectrum array for (capture, block b, variant) at this tile's Doppler index: with code-Doppler
// compensation the copy delayed by s(b, h) more samples (SearchArgs::n_shift), otherwise the only one.
template <class PA>
__device__ __forceinline__ size_t d_row(const PA &p, const TileIdx &ti, int b)
{
    const size_t bv = (size_t)((size_t)ti.cap * p.K + b) * p.nvar + ti.v;
    if (p.n_shift == 1) return bv;
    // the tile's Doppler index h; in an aided search rebuilt from (dop, v), which set_dop formed from the window base
    int h;
    if constexpr (PA::kAided) h = ti.dop * (1 + p.half_bin) + ti.v;
    else h = p.dop_lo + ti.d;
    return bv * p.n_shift + (size_t)(p.smax + code_shift(b, h, p.cd_div));
}

// The cell of a finished tile (one thread): ave_pwr = tot_pwr / L, snr = max_pwr / ave_pwr with IEEE division
// (search.cpp:493-494).
__device__ __forceinline__ void store_cell(const SearchArgs &p, int cap, int slot, int d, const Peak &tot, int L)
{
    acq_cell c;
    c.peak = tot.p;
    c.noise = __fdiv_rn(tot.sum, (float)L);   // ave_pwr = tot_pwr / i   (search.cpp:493)
    c.snr = __fdiv_rn(tot.p, c.noise);        // snr = max_pwr / ave_pwr (search.cpp:494)
    c.lag = (tot.n == 0x7fffffff) ? 0 : tot.n;
    p.cells[((size_t)cap * p.n_slots + slot) * p.n_dop + d] = c;
}

// Best-over-Doppler pick of Correlate(): max_snr = 0; for dop ascending: if (snr > max_snr) take it (search.cpp:455,495).
// One warp per (capture, sat) row: lanes stride over the Doppler cells, then a shuffle reduction that prefers the larger
// snr and, on equal snr, the lower Doppler index (what the sequential scan keeps).  A row whose snr never exceeds 0 (or
// is NaN) keeps {lag 0, dop 0, zeros}.
// Latency matters here (the pick is the tail of every small search): a warp takes ROWS rows at a time and issues ALL
// their cell loads -- whole 16-byte cells, two per lane and row, which covers 64 Doppler indices -- before it looks at
// any of them, and the winning lane hands its cell over by shuffles, so a batch costs one L2 round trip instead of
// three per row (measured with the trace variant: 1.4 us per row before, 82 rows of the all-constellation search).
template <int ROWS>
__device__ __forceinline__ void pick_rows(const acq_cell *cells, const int *__restrict__ slot_sat, acq_record *out, int row0,
                                          int row_step, int n_rows, int n_slots, int n_dop, const PickDop &pd, int lane)
{
    for (int rb = row0; rb < n_rows; rb += ROWS * row_step) {
        float4 c[ROWS][2];
#pragma unroll
        for (int i = 0; i < ROWS; i++) {
            const int row = rb + i * row_step;
#pragma unroll
            for (int j = 0; j < 2; j++) {
                const int d = lane + 32 * j;
                c[i][j] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
                if (row < n_rows && d < n_dop)
                    c[i][j] = __ldcg(reinterpret_cast<const float4 *>(cells + (size_t)row * n_dop + d));  // {peak, noise, snr, lag}
            }
        }
#pragma unroll
        for (int i = 0; i < ROWS; i++) {
            const int row = rb + i * row_step;
            if (row >= n_rows) continue;   // warp-uniform
            float4 best = c[i][0];
            int best_d = lane;
            if (!(best.z > 0.0f)) best.z = 0.0f, best_d = 0x7fffffff;           // snr > max_snr (0), NaN never wins
            if (c[i][1].z > best.z) best = c[i][1], best_d = lane + 32;         // ascending d within a lane: first maximum kept
            for (int d = lane + 64; d < n_dop; d += 32) {                        // spans beyond 64 Doppler indices
                const float4 v = __ldcg(reinterpret_cast<const float4 *>(cells + (size_t)row * n_dop + d));
                if (v.z > best.z) best = v, best_d = d;
            }
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) {
                const float s2 = __shfl_xor_sync(0xffffffffu, best.z, off);
                const int d2 = __shfl_xor_sync(0xffffffffu, best_d, off);
                const float p2 = __shfl_xor_sync(0xffffffffu, best.x, off);
                const float n2 = __shfl_xor_sync(0xffffffffu, best.y, off);
                const float l2 = __shfl_xor_sync(0xffffffffu, best.w, off);
                if (s2 > best.z || (s2 == best.z && d2 < best_d)) best = make_float4(p2, n2, s2, l2), best_d = d2;
            }
            if (lane == 0) {
                acq_record r;
                r.sat = slot_sat[row % n_slots];
                r.lag = 0;
                r.dop = 0;
                r.peak = 0.0f;
                r.noise = 0.0f;
                r.snr = 0.0f;
                if (best.z > 0.0f) {
                    r.lag = __float_as_int(best.w);
                    r.dop = (pd.dop_center ? window_lo(__ldg(pd.dop_center + row), pd.half_width, pd.dop_lo, pd.dop_hi) : pd.dop_lo) + best_d;
                    r.peak = best.x;
                    r.noise = best.y;
                    r.snr = best.z;
                }
                out[row] = r;
            }
        }
    }
}

// End of a search kernel's CTA that stored cells.  Small searches (SearchArgs::ctas_total > 0) do not wait for the
// search grids to drain before the best-Doppler pick: every cell-storing CTA bumps a counter once, after a fence, and
// k_pick_small -- launched behind the search by programmatic dependent launch, resident as soon as a search CTA has
// retired -- polls that counter instead of waiting for grid completion.  (The pick itself cannot live in the search
// kernels: ptxas balances its MOV / IMAD.MOV choice over the whole kernel, and the pick's integer code tips the hot
// loop's 40 register moves per sub-FFT onto the FMA pipe -- measured -6 % on the K = 20 kernel.)
__device__ __forceinline__ void search_cta_epilogue(const SearchArgs &p, int t)
{
    if (p.ctas_total && t == 0) {
        __threadfence();  // this CTA's cells (all stored by this thread) before the count
        atomicAdd(p.ctas_done, 1u);
    }
}

// x[a] = conj(data[k]) * code[k - dop], k = 1024 a + 4 t + k2   (search.cpp:471, support/simd.cpp:12-40).
// The Doppler shift is a pointer offset (r, q) into the margin-extended polyphase code rows.
template <class PA>
__device__ __forceinline__ void load_products(float2 (&x)[16], const PA &p, const TileIdx &ti, int b, int k2,
                                              int t)
{
    const int r = (k2 - ti.dop) & 3;
    const int q = (k2 - ti.dop - r) >> 2;
    const float2 *Dk = p.Dp + d_row(p, ti, b) * kN + k2 * kSub + t;
    const float2 *Ek = p.Ep + (size_t)(ti.sat * 4 + r) * p.ext_len + p.Q + q + t;
#pragma unroll
    for (int a = 0; a < 16; a++) x[a] = cmul_conj_a(__ldg(Dk + 256 * a), __ldg(Ek + 256 * a));
}

__device__ __forceinline__ float cpower(float2 a)
{
    const float2 sq = __fmul2_rn(a, a);
    return sq.x + sq.y;  // re^2 + im^2   (search.cpp:487)
}

// Warp-level part of the peak reduction: shuffles, then lane 0 leaves the warp's partial in `slot`.
__device__ __forceinline__ void warp_reduce_peak(Peak v, float *slot_f, int *slot_i, int t)
{
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        const float p = __shfl_xor_sync(0xffffffffu, v.p, off);
        const int n = __shfl_xor_sync(0xffffffffu, v.n, off);
        const float s = __shfl_xor_sync(0xffffffffu, v.sum, off);
        peak_merge(v, p, n, s);
    }
    const int w = t >> 5;
    if ((t & 31) == 0) {
        slot_f[w] = v.p;
        slot_f[8 + w] = v.sum;
        slot_i[w] = v.n;
    }
}

// The same with the maximum and its first index found by two warp-wide integer reductions (REDUX): powers are
// non-negative floats, so their bit patterns order like unsigned integers; among the lanes that hold the maximum the
// lowest lag wins (search.cpp:488).  The sum keeps the butterfly order of warp_reduce_peak: same bits.
__device__ __forceinline__ void warp_reduce_peak_redux(Peak v, float *slot_f, int *slot_i, int t)
{
    const unsigned pbits = __float_as_uint(v.p);
    const unsigned pmax = __reduce_max_sync(0xffffffffu, pbits);
    const unsigned nmin = __reduce_min_sync(0xffffffffu, pbits == pmax ? (unsigned)v.n : 0xffffffffu);
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) v.sum += __shfl_xor_sync(0xffffffffu, v.sum, off);
    const int w = t >> 5;
    if ((t & 31) == 0) {
        slot_f[w] = __uint_as_float(pmax);
        slot_f[8 + w] = v.sum;
        slot_i[w] = (int)nmin;
    }
}

// Merge of the eight warp partials (one thread), after a CTA barrier that follows warp_reduce_peak.
__device__ __forceinline__ Peak merge_warp_peaks(const float *slot_f, const int *slot_i)
{
    Peak v;
    v.p = slot_f[0];
    v.n = slot_i[0];
    v.sum = slot_f[8];
#pragma unroll
    for (int k = 1; k < 8; k++) peak_merge(v, slot_f[k], slot_i[k], slot_f[8 + k]);
    return v;
}

// The C/A search kernels.  Both operands of a sub-FFT are staged in shared memory by TMA bulk copies issued one
// sub-FFT ahead (see subfft4096_inv4): D into the idle half of the exchange buffer, E into its own 32 KiB buffer; the
// B->C tiles live inside the exchange rows.  The L2 round trip is off every warp's dependent chain (the load-from-L2
// A/B form, acq_variants.cuh, is 7 % slower); 98.6 KiB of shared memory per CTA, two CTAs per SM.
//
// Unroll factor of the loop over the four residues of a transform.  Rolled, the compiler moves the 16 accumulators
// between two register sets once per sub-FFT (about 40 MOVs per warp and sub-FFT in the ncu source view); unrolled
// by two it renames instead.  Measured: K = 1 kernel +1.3 % (cfg5) and -1.2 us per cold-start search (cfg1); K > 1
// kernel unchanged (27.79 M tiles/s either way), so it stays rolled; by four the kernels spill.
#ifndef ACQ_K2_UNROLL
#define ACQ_K2_UNROLL 2
#endif
constexpr int kK2Unroll = ACQ_K2_UNROLL;

// Shared prologue/epilogue state of the two C/A kernels.
struct L1Smem {
    FftSmem4 s;
    float *red_f;  // [2 parities][16], then the TMEM slot at [48]
    int *red_i;    // [2 parities][8]
};
__device__ __forceinline__ L1Smem l1_smem_carve(unsigned char *smem)
{
    L1Smem m;
    m.s = fft_smem4_carve(smem);
    m.red_f = reinterpret_cast<float *>(smem + fft_smem4_bytes());
    m.red_i = reinterpret_cast<int *>(m.red_f + 32);
    return m;
}

// max / first argmax / sum of this thread's 16 lags n = lag_of3(t, n2) < 4092 (search.cpp:486-490); n grows with n2
__device__ __forceinline__ Peak thread_peak_l1(const float (&pw)[16], int t)
{
    Peak best;
    best.p = 0.0f;
    best.n = 0x7fffffff;
    best.sum = 0.0f;
#pragma unroll
    for (int n2 = 0; n2 < 16; n2++) {
        const int n = lag_of3(t, n2);
        if (n2 < 15 || n < ACQ_LAGS_L1) {
            if (pw[n2] > best.p) best.p = pw[n2], best.n = n;
            best.sum += pw[n2];
        }
    }
    return best;
}

// k_search_l1<MULTI> -- persistent CTAs (two per SM) stride over the tiles.  MULTI (k_noncoh > 1): a tile runs K
// inverse FFTs whose powers are summed in registers, P[n] += |r_b[(n + 16 b) mod N]|^2; the 16-lag-per-block code
// advance is removed in the front end by delaying block b (see k_hb2).
// (Tried in round 2 and dropped: a K = 1 form that cuts the 4 n_tiles sub-FFT units into equal contiguous ranges per
// CTA and hands the partial accumulators of a split tile over through L2 -- "stream-K" -- so that 1312 tiles do not
// run as five rounds on 296 CTAs.  Bitwise-equal cells, but 78.6 -> 81.4 us per cold-start search and no change on
// the receiver farm: the last round already runs one CTA per SM, which is 1.6x faster per tile than two.)
#ifndef ACQ_L1_LEAN
#define ACQ_L1_LEAN 1   // K = 1: tile indices advance without divisions, max / first index by REDUX (+0.3..1 % cfg5, -1.3 us cfg1; 0 = round-1 form)
#endif
template <bool MULTI, class PA>
__global__ void __launch_bounds__(256, 2) k_search_l1(const PA p)
{
    extern __shared__ __align__(1024) unsigned char smem[];
    const L1Smem m = l1_smem_carve(smem);
    const FftSmem4 &s = m.s;
    float *red_f = m.red_f;
    int *red_i = m.red_i;
    const int t = threadIdx.x;
    ACQ_TRACE_STAMP(kTrSearchL1, 0);
    constexpr int L = ACQ_LAGS_L1;
    const uint32_t tmem_base = tmem_alloc_cta<2 * kTwCols>(reinterpret_cast<uint32_t *>(red_f + 48), t);
    const uint32_t tw_taddr = tmem_base + tmem_lane_base(t) + (uint32_t)((t >> 7) * kTwCols);
    subfft4_park_twiddles(p.tables, tw_taddr, t);
    float2 bw = __ldg(p.tables + kT2Elems + t);  // W16384^{4t}: base of residue 0; later bases come from TMEM
    const uint32_t bar = smem_u32(s.bar);
    if (t == 0) mbar_init(bar, 1);
    __syncthreads();
    if (p.wait_prior) pdl_wait();
    ACQ_TRACE_STAMP(kTrSearchL1, 1);
    pdl_trigger_search();
    // thread 0: stage the operands of sub-FFT (tn, bn, k2n) -- D into S1 half `half`, E into the E buffer
    auto issue = [&](const TileIdx &tn, int bn, int k2n, int half) {
        const int r = (k2n - tn.dop) & 3;
        const int q = (k2n - tn.dop - r) >> 2;
#ifdef ACQ_KO_SAME_OPERANDS  // knock-out experiment (wrong results): every tile reads the same 64 KiB of operands
        const float2 *Dk = p.Dp + k2n * kSub;
        const float2 *Ek = p.Ep + (size_t)r * p.ext_len + ((p.Q + q) & ~1);
#else
        const float2 *Dk = p.Dp + d_row(p, tn, bn) * kN + k2n * kSub;
        const float2 *Ek = p.Ep + (size_t)(tn.sat * 4 + r) * p.ext_len + ((p.Q + q) & ~1);
#endif
        fence_proxy_async();  // generic-proxy reads of these buffers (ordered by the CTA barrier) before the async writes
#ifdef ACQ_K1_E_LDG   // experiment: the code run straight from L2 (issued before the wait for D), only D staged
        (void)Ek;
        mbar_expect_tx(bar, (uint32_t)(sizeof(float2) * kSub));
#else
        mbar_expect_tx(bar, (uint32_t)(sizeof(float2) * (kSub + kEBufElems)));
        tma_load_1d(smem_u32(s.E), Ek, (uint32_t)(sizeof(float2) * kEBufElems), bar);
#endif
        tma_load_1d(smem_u32(s.S1 + half * kS1pElems), Dk, (uint32_t)(sizeof(float2) * kSub), bar);
    };
    TileIdx ti(p, blockIdx.x);   // the grid never exceeds the tile count: every CTA has a first tile
    if (t == 0) issue(ti, 0, 0, 0);
    int *feed = red_i + 20;      // dynamic tile feed (claim_tile / publish_tile / next_tile)
    unsigned nxt = blockIdx.x;   // thread 0: the tile being run, then the claimed one
    int it = 0;  // sub-FFT counter: S1 half and mbarrier phase parity = it & 1
    int par = 0, pend_cap = -1, pend_slot = 0, pend_d = 0;
    // The cross-warp merge of a tile's peak is deferred to the next tile: the warp partials are left in a parity slot
    // and thread 0 merges them after the next tile's first sub-FFT barrier, so the reduction costs no CTA barrier of
    // its own (it matters at K = 1, where a tile is only four sub-FFTs).
    auto flush = [&]() {
        store_cell(p, pend_cap, pend_slot, pend_d, merge_warp_peaks(red_f + 16 * (par ^ 1), red_i + 8 * (par ^ 1)), L);
    };

    for (;;) {
        float P[16];
        float2 acc[16];
        for (int b = 0; b < p.K; b++) {
            float2 x[16];
            constexpr int kUnroll = MULTI ? 1 : kK2Unroll;
#pragma unroll kUnroll
            for (int k2 = 0; k2 < 4; k2++) {
                float2 *S1b = s.S1 + (it & 1) * kS1pElems;
                {   // x[a] = conj(data[k]) * code[k - dop], k = 1024 a + 4 t + k2   (search.cpp:471), operands from smem
                    const int r = (k2 - ti.dop) & 3;
                    const int q = (k2 - ti.dop - r) >> 2;
                    const float2 *Dk = S1b + t;
#ifdef ACQ_K1_E_LDG
                    const float2 *Eg = p.Ep + (size_t)(ti.sat * 4 + r) * p.ext_len + p.Q + q + t;
#pragma unroll
                    for (int a = 0; a < 16; a++) x[a] = __ldg(Eg + 256 * a);
                    mbar_wait(bar, (uint32_t)(it & 1));
#pragma unroll
                    for (int a = 0; a < 16; a++) x[a] = cmul_conj_a(Dk[kRowElems * a], x[a]);
#else
                    const float2 *Ek = s.E + ((p.Q + q) & 1) + t;
                    mbar_wait(bar, (uint32_t)(it & 1));
#pragma unroll
                    for (int a = 0; a < 16; a++) x[a] = cmul_conj_a(Dk[kRowElems * a], Ek[256 * a]);
#endif
                }
                subfft4096_inv4<true>(x, k2, bw, S1b, t, tw_taddr, [&]() {
                    if (t == 0) {  // every warp is past its operand reads of this sub-FFT and past stage C of the previous one
                        if (b == 0 && k2 == 0) nxt = claim_tile(p, nxt);
                        if (b == p.K - 1 && k2 == 2) publish_tile(feed, p, nxt);
                        if (k2 < 3) issue(ti, b, k2 + 1, (it + 1) & 1);
                        else if (b + 1 < p.K) issue(ti, b + 1, 0, (it + 1) & 1);
                        else {
                            TileIdx tn;
                            if (next_tile(feed, tn)) issue(tn, 0, 0, (it + 1) & 1);
                        }
                    }
                });
                it++;
                if (t == 0 && b == 0 && k2 == 0 && pend_cap >= 0) flush();
                if (k2 == 0) {
#pragma unroll
                    for (int n2 = 0; n2 < 16; n2++) acc[n2] = x[r16(n2)];
                } else {
#pragma unroll
                    for (int n2 = 0; n2 < 16; n2++) acc[n2] = cfma(x[r16(n2)], c_cC[k2][n2], acc[n2]);
                }
            }
            // block b was delayed by 16*b samples in the front end (k_front_end), so lag n lines up across blocks
#pragma unroll
            for (int n2 = 0; n2 < 16; n2++) P[n2] = (!MULTI || b == 0) ? cpower(acc[n2]) : (P[n2] + cpower(acc[n2]));
        }
#if ACQ_L1_LEAN
        warp_reduce_peak_redux(thread_peak_l1(P, t), red_f + 16 * par, red_i + 8 * par, t);
#else
        warp_reduce_peak(thread_peak_l1(P, t), red_f + 16 * par, red_i + 8 * par, t);
#endif
        pend_cap = ti.cap;
        pend_slot = ti.slot;
        pend_d = ti.d;
        par ^= 1;
        if (!next_tile(feed, ti)) break;   // published behind the barrier of sub-FFT 2, read behind that of sub-FFT 3
    }
    __syncthreads();
    if (t == 0 && pend_cap >= 0) flush();
    claims_done(p, t);
    search_cta_epilogue(p, t);
    ACQ_TRACE_STAMP(kTrSearchL1, 2);
    tmem_free_cta<2 * kTwCols>(tmem_base, t);
}

// Staging warps (k_search_l1_dr below; measured first in the experiment form k_search_l1_st, acq_variants.cuh).  In
// k_search_l1 thread 0 of a CTA issues the next sub-FFT's bulk copies right after the CTA barrier (address arithmetic, proxy
// fence, expect_tx, the copies) and once per tile merges the warp partials and stores the cell: ncu's warp samples put a
// third of a sub-FFT period of warp 0 on that path, and the other seven warps wait for it at the next barrier (10 % of all
// warp samples were barrier stalls).  Here one CTA per SM holds TWO teams of eight FFT warps -- each team is what a CTA
// of k_search_l1 is, with its own exchange and code-run buffers, mbarrier, tensor-memory columns and named barrier -- plus
// one staging warp per team that takes part in the team's barrier and does all of the above, so no FFT warp ever leaves
// the common instruction stream.  Five warpgroups: the launch allocates 96 registers per thread, the staging warpgroup
// drops to 32 (setmaxnreg.dec) and the four FFT warpgroups rise to 112 with exactly what it released.
[[maybe_unused]] constexpr int kStThreads = 640, kStHandOver = 288;   // 2 x 256 FFT threads + a warpgroup of staging warps; hand-over = 8 + 1 warps
// Named barriers of a team (ids 1..3 for team 0, 4..6 for team 1):
//   A (256 threads): the FFT warps' own barrier, one per sub-FFT;
//   B (288): hand-over to the staging warp.  Every FFT warp ARRIVES (no wait) just before it waits on A, and the staging
//      warp SYNCs: it runs on once all eight have reached this sub-FFT's barrier, i.e. are past their operand reads of this
//      sub-FFT and past stage C of the one before, and stages the next sub-FFT's operands.  An FFT warp cannot reach the
//      next sub-FFT's barrier before the staging warp has passed (that sub-FFT's operands are staged only after it), so
//      the phases of B cannot mix;
//   C (288): the same hand-over once more after a team's last sub-FFT (the last tile's warp partials are in place).
// All waiting participants of a barrier execute the same instruction: compute-sanitizer's synccheck rejects a bar.sync
// reached from two code locations (tools/exp/mb_namedbar.cu), which rules out the simplest form -- the staging warp inside
// barrier A, one barrier instruction per FFT warp: 5.84 ms on cfg5 with 128 captures, against 5.97 ms for this form,
// 6.02 ms with the arrive moved up behind the products, 6.18 ms with one warp arriving after A, 6.29 ms with the staging
// warp polling a shared-memory mbarrier, and 6.30 ms for k_search_l1<false>.
__device__ __forceinline__ void st_fft_sync(int team)         // barrier A
{
    if (team == 0) asm volatile("bar.sync 1, 256;" ::: "memory");
    else asm volatile("bar.sync 4, 256;" ::: "memory");
}
__device__ __forceinline__ void st_fft_arrive(int team)       // barrier B, FFT warps
{
    if (team == 0) asm volatile("bar.arrive 2, %0;" ::"n"(kStHandOver) : "memory");
    else asm volatile("bar.arrive 5, %0;" ::"n"(kStHandOver) : "memory");
}
__device__ __forceinline__ void st_fft_done(int team)         // barrier C, FFT warps
{
    if (team == 0) asm volatile("bar.arrive 3, %0;" ::"n"(kStHandOver) : "memory");
    else asm volatile("bar.arrive 6, %0;" ::"n"(kStHandOver) : "memory");
}
__device__ __forceinline__ void st_stage_wait(int team)       // barrier B, staging warp
{
    if (team == 0) asm volatile("bar.sync 2, %0;" ::"n"(kStHandOver) : "memory");
    else asm volatile("bar.sync 5, %0;" ::"n"(kStHandOver) : "memory");
}
__device__ __forceinline__ void st_stage_wait_done(int team)  // barrier C, staging warp
{
    if (team == 0) asm volatile("bar.sync 3, %0;" ::"n"(kStHandOver) : "memory");
    else asm volatile("bar.sync 6, %0;" ::"n"(kStHandOver) : "memory");
}

// k_search_l1_dr -- the staging-warp form with the CAPTURE operand resident in tensor memory.  The capture residue D of a
// sub-FFT depends on (capture, residue k2) only, and a thread always reads the same 16 values of it (D[256 a + t]):
// 4 residues x 16 complex = the 128 TMEM columns a thread owns.  A team takes a CONTIGUOUS range of tiles (capture-major
// order: all (satellite, Doppler) tiles of a capture are neighbours), so D is staged by TMA and parked only in the first
// tile of a capture and comes back by one tcgen05.ld per sub-FFT in every other tile: neither its 32 KiB bulk copy nor its 16
// shared-memory loads per thread touch the L1/shared data pipe.  The stage-B twiddles move to a 7.5 KiB shared table per
// team, the stage-A bases to the global table (as in k_search_l1_multi).  Same arithmetic in the same order as
// k_search_l1<false>: bitwise-equal cells (tested).
struct DrSmem {
    float2 *S1;  // [2][4096]
    float2 *E;   // [4098]
    unsigned long long *bar;
    float2 *T2;  // [4][15][16]
    float *red_f;
    int *red_i;
};
__host__ __device__ constexpr size_t dr_team_smem_bytes()
{
    return (sizeof(float2) * (size_t)(2 * kSub + kEBufElems) + 16 + sizeof(float2) * kT2Elems + 64 * sizeof(float) + 1023) / 1024 * 1024;
}
__host__ __device__ constexpr size_t dr_smem_bytes() { return 2 * dr_team_smem_bytes(); }
__device__ __forceinline__ DrSmem dr_smem_carve(unsigned char *smem)
{
    DrSmem s;
    s.S1 = reinterpret_cast<float2 *>(smem);
    s.E = s.S1 + 2 * kSub;
    s.bar = reinterpret_cast<unsigned long long *>(s.E + kEBufElems);
    s.T2 = reinterpret_cast<float2 *>(s.bar + 2);
    s.red_f = reinterpret_cast<float *>(s.T2 + kT2Elems);
    s.red_i = reinterpret_cast<int *>(s.red_f + 32);
    return s;
}

// Compiled only into the variant libraries that route searches to it (l1_dr_all, l1_dr12): the product library holds no
// A/B kernel.
#ifndef ACQ_DR_MIN_TILES_PER_SM
#define ACQ_DR_MIN_TILES_PER_SM -1   // product: never (see search_kind_l1)
#endif
#if ACQ_DR_MIN_TILES_PER_SM >= 0
__global__ void __launch_bounds__(kStThreads, 1) k_search_l1_dr(const SearchArgs p)
{
    extern __shared__ __align__(1024) unsigned char smem[];
    const int t = threadIdx.x;
    ACQ_TRACE_STAMP(kTrSearchL1, 0);
    constexpr int L = ACQ_LAGS_L1;
    __shared__ uint32_t tmem_slot;
    const uint32_t tmem_base = tmem_alloc_cta<4 * kTwCols>(&tmem_slot, t);
    if (t < 2) mbar_init(smem_u32(dr_smem_carve(smem + t * dr_team_smem_bytes()).bar), 1);
    __syncthreads();
    if (p.wait_prior) pdl_wait();
    ACQ_TRACE_STAMP(kTrSearchL1, 1);
    pdl_trigger_search();
    // Team T of 2 gridDim.x takes the T-th of as many balanced contiguous tile ranges (team 1 of a CTA comes after every
    // team 0: a search of no more tiles than SMs runs one team per SM).
    const int team = (t < 512) ? (t >> 8) : ((t >> 5) & 1);
    const unsigned T = (unsigned)team * gridDim.x + blockIdx.x, n_teams = 2u * gridDim.x;
    const unsigned n_tiles = (unsigned)p.n_tiles, base = n_tiles / n_teams, extra = n_tiles % n_teams;
    const unsigned tile0 = T * base + (T < extra ? T : extra), my_tiles = base + (T < extra ? 1u : 0u);
    const unsigned per_cap = (unsigned)p.n_work * (unsigned)p.n_dop;   // tiles of one capture
    const DrSmem s = dr_smem_carve(smem + team * dr_team_smem_bytes());
    const uint32_t bar = smem_u32(s.bar);
    if (t >= 512) {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 32;");
        if (t < 576 && my_tiles > 0) {
            // ---- staging warp of `team` (lane 0 works)
            const bool lead = (t & 31) == 0;
            float *red_f = s.red_f;
            int *red_i = s.red_i;
            auto issue = [&](const TileIdx &tn, bool fresh, int k2n, int half) {   // E always, D in the first tile of a capture
                const int r = (k2n - tn.dop) & 3;
                const int q = (k2n - tn.dop - r) >> 2;
                const float2 *Ek = p.Ep + (size_t)(tn.sat * 4 + r) * p.ext_len + ((p.Q + q) & ~1);
                fence_proxy_async();  // generic-proxy accesses of these buffers (ordered by the team barrier) before the async writes
                mbar_expect_tx(bar, (uint32_t)(sizeof(float2) * (kEBufElems + (fresh ? kSub : 0))));
                tma_load_1d(smem_u32(s.E), Ek, (uint32_t)(sizeof(float2) * kEBufElems), bar);
                if (fresh) {
                    const float2 *Dk = p.Dp + d_row(p, tn, 0) * kN + k2n * kSub;
                    tma_load_1d(smem_u32(s.S1 + half * kSub), Dk, (uint32_t)(sizeof(float2) * kSub), bar);
                }
            };
            TileIdx ti(p, tile0);
            bool fresh = true;
            if (lead) issue(ti, true, 0, 0);
            int it = 0, par = 0, pend_cap = -1, pend_slot = 0, pend_d = 0;
            for (unsigned i = 0; i < my_tiles; i++) {
                TileIdx tn = ti;
                const bool more = i + 1 < my_tiles;
                if (more) tn.step(p, 1, 0, 0);
                const bool fresh_n = tn.cap != ti.cap;
#pragma unroll 1
                for (int k2 = 0; k2 < 4; k2++) {
                    __syncwarp();
                    st_stage_wait(team);   // every FFT warp is past its operand reads of this sub-FFT and past stage C of the previous one
                    if (lead) {
                        if (k2 < 3) issue(ti, fresh, k2 + 1, (it + 1) & 1);
                        else if (more) issue(tn, fresh_n, 0, (it + 1) & 1);
                        if (k2 == 0 && pend_cap >= 0)   // the previous tile's peak: its warp partials precede this barrier
                            store_cell(p, pend_cap, pend_slot, pend_d, merge_warp_peaks(red_f + 16 * (par ^ 1), red_i + 8 * (par ^ 1)), L);
                    }
                    it++;
                }
                pend_cap = ti.cap;
                pend_slot = ti.slot;
                pend_d = ti.d;
                par ^= 1;
                ti = tn;
                fresh = fresh_n;
            }
            __syncwarp();
            st_stage_wait_done(team);   // the last tile's warp partials are in place
            if (lead) {
                store_cell(p, pend_cap, pend_slot, pend_d, merge_warp_peaks(red_f + 16 * (par ^ 1), red_i + 8 * (par ^ 1)), L);
                __threadfence();  // this team's cells (all stored by this thread) before the CTA's count
#ifdef ACQ_TRACE
                if (blockIdx.x < kTraceCtas) {   // slot 3: team 0 done; team 1 done goes to the second half of the CTA axis
                    unsigned long long tm;
                    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(tm));
                    g_trace[kTrSearchL1][blockIdx.x + (team ? 512 : 0)][3] = tm;
                }
#endif
            }
        }
    } else {
        asm volatile("setmaxnreg.inc.sync.aligned.u32 112;");
        if (my_tiles > 0) {
            // ---- the eight FFT warps of `team`
            const int tt = t & 255;
            float *red_f = s.red_f;
            int *red_i = s.red_i;
            const uint32_t d_taddr = tmem_base + (uint32_t)(team * 2 * kTwCols) + tmem_lane_base(tt) + (uint32_t)((tt >> 7) * kTwCols);  // [k2][16 complex]
            {   // stage-B twiddle table into this team's shared memory
                const float4 *src = reinterpret_cast<const float4 *>(p.tables);
                float4 *dst = reinterpret_cast<float4 *>(s.T2);
                for (int i = tt; i < kT2Elems / 2; i += 256) dst[i] = __ldg(src + i);
            }
            const float2 *bases = p.tables + kT2Elems + tt;  // [k2][256]: W16384^{4t+k2}
            float2 bw = __ldg(bases);
            int it = 0, par = 0;
            const TileIdx t0(p, tile0);
            int d = t0.d, dop = t0.dop;
            unsigned left = per_cap - tile0 % per_cap;   // tiles of this team's range before the next capture begins
            bool fresh = true;
            st_fft_sync(team);   // the twiddle table is in place
            for (unsigned i = 0; i < my_tiles; i++) {
                float P[16];
                float2 acc[16];
                float2 x[16];
                // rolled: at 112 registers the loop unrolled by two spills (28.75 M against 27.7 M tiles/s on cfg5, measured)
#pragma unroll 1
                for (int k2 = 0; k2 < 4; k2++) {
                    float2 *S1b = s.S1 + (it & 1) * kSub;
                    const int r = (k2 - dop) & 3;
                    const int q = (k2 - dop - r) >> 2;
                    const float2 *Ek = s.E + ((p.Q + q) & 1) + tt;
                    if (fresh) {   // D from the staged residue; park this thread's 16 values for the capture's other tiles
                        const float2 *Dk = S1b + tt;
                        mbar_wait(bar, (uint32_t)(it & 1));
#pragma unroll
                        for (int a = 0; a < 16; a++) x[a] = Dk[256 * a];
                        tmem_st16(d_taddr + 32 * k2, x);
                        tmem_wait_st();
                    } else {
                        tmem_ld16(d_taddr + 32 * k2, x);
                        mbar_wait(bar, (uint32_t)(it & 1));
                        tmem_wait_ld();
                    }
                    // x[a] = conj(data[k]) * code[k - dop], k = 1024 a + 4 t + k2   (search.cpp:471)
#pragma unroll
                    for (int a = 0; a < 16; a++) x[a] = cmul_conj_a(x[a], Ek[256 * a]);
                    subfft4096_inv4s(x, k2, bw, S1b, tt, s.T2, BaseFromGlobal{bases}, [&] { st_fft_arrive(team); st_fft_sync(team); }, [] {});
                    it++;
                    if (k2 == 0) {
#pragma unroll
                        for (int n2 = 0; n2 < 16; n2++) acc[n2] = x[r16(n2)];
                    } else {
#pragma unroll
                        for (int n2 = 0; n2 < 16; n2++) acc[n2] = cfma(x[r16(n2)], c_cC[k2][n2], acc[n2]);
                    }
                }
#pragma unroll
                for (int n2 = 0; n2 < 16; n2++) P[n2] = cpower(acc[n2]);
                warp_reduce_peak_redux(thread_peak_l1(P, tt), red_f + 16 * par, red_i + 8 * par, tt);
                par ^= 1;
                {   // next tile of the range: the Doppler index (the only tile coordinate an FFT warp needs) and the capture boundary
                    if (++d >= p.n_dop) d = 0;
                    const int h = p.dop_lo + d;
                    const int v = p.half_bin ? (h & 1) : 0;
                    dop = p.half_bin ? ((h - v) >> 1) : h;
                    fresh = (--left == 0);
                    if (fresh) left = per_cap;
                }
            }
            st_fft_done(team);   // the last tile's warp partials are in place
        }
    }
    __syncthreads();
    if (t == 0 && p.ctas_total) atomicAdd(p.ctas_done, 1u);   // both teams' cells are stored and fenced (staging warps, above)
    ACQ_TRACE_STAMP(kTrSearchL1, 2);
    tmem_free_cta<4 * kTwCols>(tmem_base, t);
}
#endif  // ACQ_DR_MIN_TILES_PER_SM >= 0


// k_search_l1_multi -- k_noncoh > 1 with the CODE operand resident in tensor memory.  The code run E of a tile depends on
// (satellite, Doppler, residue k2) but not on the block b, and a thread always reads the same 16 values of it
// (E[256 a + t]): 4 residues x 16 complex = exactly the 128 TMEM columns a thread owns.  They are staged by TMA and
// parked during block 0 and come back by one tcgen05.ld per sub-FFT for blocks 1..K-1 -- 19 of 20 in cfg2 -- so for those
// neither the 32 KiB bulk copy of E nor its 16 shared-memory loads per thread touch the L1/shared data pipe, the
// kernel's busiest unit (-20 % wavefronts per tile).  The stage-B twiddles, which k_search_l1<true> keeps in those
// columns, move to a 7.5 KiB shared-memory table (15 broadcast loads per thread and sub-FFT: +6 %), the stage-A bases to
// the 8 KiB global table (L1-resident).  106 KiB of shared memory per CTA, two CTAs per SM; same arithmetic in the same
// order as k_search_l1<true>, so the cells are bitwise equal (tested against the variant that keeps the old form).
struct L1MultiSmem {
    float2 *S1;  // [2][4096]
    float2 *E;   // [4098]
    unsigned long long *bar;
    float2 *T2;  // [4][15][16]
    float *red_f;
    int *red_i;
};
__host__ __device__ constexpr size_t l1_multi_smem_bytes()
{
    return sizeof(float2) * (size_t)(2 * kSub + kEBufElems) + 16 + sizeof(float2) * kT2Elems + 64 * sizeof(float);
}

// Residue loop fully unrolled (24 bytes of spill): cfg2 3.53 ms rolled, 3.33 ms by two, 3.21 ms by four on one box, with
// claimed tiles.  (On the static stride, earlier in round 2, the factor made no difference: the slower CTA of each SM
// set the pace.)
#ifndef ACQ_MULTI_UNROLL
#define ACQ_MULTI_UNROLL 4
#endif
template <class PA>
__global__ void __launch_bounds__(256, 2) k_search_l1_multi(const PA p)
{
    extern __shared__ __align__(1024) unsigned char smem[];
    L1MultiSmem s;
    s.S1 = reinterpret_cast<float2 *>(smem);
    s.E = s.S1 + 2 * kSub;
    s.bar = reinterpret_cast<unsigned long long *>(s.E + kEBufElems);
    s.T2 = reinterpret_cast<float2 *>(s.bar + 2);
    s.red_f = reinterpret_cast<float *>(s.T2 + kT2Elems);  // [2 parities][16], then the TMEM slot at [48]
    s.red_i = reinterpret_cast<int *>(s.red_f + 32);        // [2 parities][8]
    float *red_f = s.red_f;
    int *red_i = s.red_i;
    const int t = threadIdx.x;
    ACQ_TRACE_STAMP(kTrSearchL1, 0);
    constexpr int L = ACQ_LAGS_L1;
    const uint32_t tmem_base = tmem_alloc_cta<2 * kTwCols>(reinterpret_cast<uint32_t *>(red_f + 48), t);
    const uint32_t e_taddr = tmem_base + tmem_lane_base(t) + (uint32_t)((t >> 7) * kTwCols);  // [k2][16 complex]
    {   // stage-B twiddle table into shared memory
        const float4 *src = reinterpret_cast<const float4 *>(p.tables);
        float4 *dst = reinterpret_cast<float4 *>(s.T2);
        for (int i = t; i < kT2Elems / 2; i += 256) dst[i] = __ldg(src + i);
    }
    const float2 *bases = p.tables + kT2Elems + t;  // [k2][256]: W16384^{4t+k2}
    float2 bw = __ldg(bases);
    const uint32_t bar = smem_u32(s.bar);
    if (t == 0) mbar_init(bar, 1);
    __syncthreads();
    if (p.wait_prior) pdl_wait();
    ACQ_TRACE_STAMP(kTrSearchL1, 1);
    pdl_trigger_search();
    // thread 0: stage the operands of sub-FFT (tn, bn, k2n) -- D into S1 half `half`; E only for block 0
    auto issue = [&](const TileIdx &tn, int bn, int k2n, int half) {
        const int r = (k2n - tn.dop) & 3;
        const int q = (k2n - tn.dop - r) >> 2;
        const float2 *Dk = p.Dp + d_row(p, tn, bn) * kN + k2n * kSub;
        fence_proxy_async();  // generic-proxy reads of these buffers (ordered by the CTA barrier) before the async writes
        if (bn == 0) {
            const float2 *Ek = p.Ep + (size_t)(tn.sat * 4 + r) * p.ext_len + ((p.Q + q) & ~1);
            mbar_expect_tx(bar, (uint32_t)(sizeof(float2) * (kSub + kEBufElems)));
            tma_load_1d(smem_u32(s.E), Ek, (uint32_t)(sizeof(float2) * kEBufElems), bar);
        } else {
            mbar_expect_tx(bar, (uint32_t)(sizeof(float2) * kSub));
        }
        tma_load_1d(smem_u32(s.S1 + half * kSub), Dk, (uint32_t)(sizeof(float2) * kSub), bar);
    };
    TileIdx ti(p, blockIdx.x);   // the grid never exceeds the tile count: every CTA has a first tile
    if (t == 0) issue(ti, 0, 0, 0);
    int *feed = red_i + 20;      // dynamic tile feed (claim_tile / publish_tile / next_tile)
    unsigned nxt = blockIdx.x;   // thread 0: the tile being run, then the claimed one
    int it = 0;  // sub-FFT counter: S1 half and mbarrier phase parity = it & 1
    int par = 0, pend_cap = -1, pend_slot = 0, pend_d = 0;
    auto flush = [&]() {   // thread 0: the previous tile's peak (deferred cross-warp merge, see k_search_l1)
        store_cell(p, pend_cap, pend_slot, pend_d, merge_warp_peaks(red_f + 16 * (par ^ 1), red_i + 8 * (par ^ 1)), L);
    };

    for (;;) {
        float P[16];
        float2 acc[16];
        for (int b = 0; b < p.K; b++) {
            float2 x[16];
            // aided: by two, which does not spill (at four the window code takes the spill from 24 to 56 bytes)
            constexpr int kMultiUnroll = PA::kAided ? 2 : ACQ_MULTI_UNROLL;
#pragma unroll kMultiUnroll
            for (int k2 = 0; k2 < 4; k2++) {
                float2 *S1b = s.S1 + (it & 1) * kSub;
                const float2 *Dk = S1b + t;
                if (b == 0) {   // E from the staged run; park this thread's 16 values for the blocks to come
                    const int r = (k2 - ti.dop) & 3;
                    const int q = (k2 - ti.dop - r) >> 2;
                    const float2 *Ek = s.E + ((p.Q + q) & 1) + t;
                    mbar_wait(bar, (uint32_t)(it & 1));
#pragma unroll
                    for (int a = 0; a < 16; a++) x[a] = Ek[256 * a];
                    tmem_st16(e_taddr + 32 * k2, x);
                    tmem_wait_st();
                } else {
                    tmem_ld16(e_taddr + 32 * k2, x);
                    mbar_wait(bar, (uint32_t)(it & 1));
                    tmem_wait_ld();
                }
                // x[a] = conj(data[k]) * code[k - dop], k = 1024 a + 4 t + k2   (search.cpp:471)
#pragma unroll
                for (int a = 0; a < 16; a++) x[a] = cmul_conj_a(Dk[256 * a], x[a]);
                subfft4096_inv4s(x, k2, bw, S1b, t, s.T2, BaseFromGlobal{bases}, [&]() {
                    if (t == 0) {  // every warp is past its operand reads of this sub-FFT and past stage C of the previous one
                        if (b == 0 && k2 == 0) nxt = claim_tile(p, nxt);
                        if (b == p.K - 1 && k2 == 2) publish_tile(feed, p, nxt);
                        if (k2 < 3) issue(ti, b, k2 + 1, (it + 1) & 1);
                        else if (b + 1 < p.K) issue(ti, b + 1, 0, (it + 1) & 1);
                        else {
                            TileIdx tn;
                            if (next_tile(feed, tn)) issue(tn, 0, 0, (it + 1) & 1);
                        }
                    }
                });
                it++;
                if (t == 0 && b == 0 && k2 == 0 && pend_cap >= 0) flush();
                if (k2 == 0) {
#pragma unroll
                    for (int n2 = 0; n2 < 16; n2++) acc[n2] = x[r16(n2)];
                } else {
#pragma unroll
                    for (int n2 = 0; n2 < 16; n2++) acc[n2] = cfma(x[r16(n2)], c_cC[k2][n2], acc[n2]);
                }
            }
            // block b was delayed by 16*b samples in the front end (k_front_end), so lag n lines up across blocks
#pragma unroll
            for (int n2 = 0; n2 < 16; n2++) P[n2] = (b == 0) ? cpower(acc[n2]) : (P[n2] + cpower(acc[n2]));
        }
        warp_reduce_peak(thread_peak_l1(P, t), red_f + 16 * par, red_i + 8 * par, t);
        pend_cap = ti.cap;
        pend_slot = ti.slot;
        pend_d = ti.d;
        par ^= 1;
        if (!next_tile(feed, ti)) break;   // published behind the barrier of the second-to-last sub-FFT, read behind the last
    }
    __syncthreads();
    if (t == 0 && pend_cap >= 0) flush();
    claims_done(p, t);
    search_cta_epilogue(p, t);
    ACQ_TRACE_STAMP(kTrSearchL1, 2);
    tmem_free_cta<2 * kTwCols>(tmem_base, t);
}

// k_search_l1_cr -- K = 1 on full bins with the CAPTURE operand resident in tensor memory and tiles claimed in CHUNKS.
// The idea of k_search_l1_dr (a thread always reads the same 16 values of a capture residue: 4 residues x 16 complex = its
// 128 TMEM columns, so D is staged and parked once and comes back by one tcgen05.ld per sub-FFT) in the two-CTAs-per-SM
// form that claims its work: a CTA draws runs of consecutive tiles (same capture, bar the boundaries), 16 tiles long while
// the launch is young, 4 and then single tiles towards its end (SearchArgs::ck_n16 / ck_n4, search_chunks()), so the
// greedy tail stays one tile long while D is re-staged for ~1 tile in 14.  Stage-B twiddles: the 7.5 KiB shared table;
// stage-A bases: the global table (as k_search_l1_multi, whose shared-memory layout this kernel uses).  Same arithmetic in
// the same order as k_search_l1<false>: bitwise-equal cells (tested).
#ifndef ACQ_CK_BIG
#define ACQ_CK_BIG 16
#endif
#ifndef ACQ_CK_MID
#define ACQ_CK_MID 4
#endif
constexpr unsigned kCkBig = ACQ_CK_BIG, kCkMid = ACQ_CK_MID;   // chunk lengths (SearchArgs::ck_n16 counts the big ones, ck_n4 the middle ones)
__device__ __forceinline__ bool chunk_of(const SearchArgs &p, unsigned c, unsigned &start, unsigned &len)
{
    if (c < p.ck_n16) {
        start = kCkBig * c, len = kCkBig;
        return true;
    }
    c -= p.ck_n16;
    if (c < p.ck_n4) {
        start = kCkBig * p.ck_n16 + kCkMid * c, len = kCkMid;
        return true;
    }
    c -= p.ck_n4;
    start = kCkBig * p.ck_n16 + kCkMid * p.ck_n4 + c, len = 1u;
    return start < (unsigned)p.n_tiles;
}

// Residue loop fully unrolled (126 registers, no spill): on a 128-capture farm 5.98 ms rolled, 5.49 ms by two, 5.24 ms by
// four (28.1 / 30.6 / 32.1 M tiles/s; k_search_l1<false> with claimed tiles: 5.78 ms, k_search_l1_dr: 5.96 ms).
#ifndef ACQ_CR_UNROLL
#define ACQ_CR_UNROLL 4
#endif
template <class PA>
__global__ void __launch_bounds__(256, 2) k_search_l1_cr(const PA p)
{
    extern __shared__ __align__(1024) unsigned char smem[];
    L1MultiSmem s;
    s.S1 = reinterpret_cast<float2 *>(smem);
    s.E = s.S1 + 2 * kSub;
    s.bar = reinterpret_cast<unsigned long long *>(s.E + kEBufElems);
    s.T2 = reinterpret_cast<float2 *>(s.bar + 2);
    s.red_f = reinterpret_cast<float *>(s.T2 + kT2Elems);  // [2 parities][16], then the TMEM slot at [48]
    s.red_i = reinterpret_cast<int *>(s.red_f + 32);        // [2 parities][8]
    float *red_f = s.red_f;
    int *red_i = s.red_i;
    const int t = threadIdx.x;
    ACQ_TRACE_STAMP(kTrSearchL1, 0);
    constexpr int L = ACQ_LAGS_L1;
    const uint32_t tmem_base = tmem_alloc_cta<2 * kTwCols>(reinterpret_cast<uint32_t *>(red_f + 48), t);
    const uint32_t d_taddr = tmem_base + tmem_lane_base(t) + (uint32_t)((t >> 7) * kTwCols);  // [k2][16 complex]
    {   // stage-B twiddle table into shared memory
        const float4 *src = reinterpret_cast<const float4 *>(p.tables);
        float4 *dst = reinterpret_cast<float4 *>(s.T2);
        for (int i = t; i < kT2Elems / 2; i += 256) dst[i] = __ldg(src + i);
    }
    const float2 *bases = p.tables + kT2Elems + t;  // [k2][256]: W16384^{4t+k2}
    float2 bw = __ldg(bases);
    const uint32_t bar = smem_u32(s.bar);
    if (t == 0) mbar_init(bar, 1);
    __syncthreads();
    if (p.wait_prior) pdl_wait();
    ACQ_TRACE_STAMP(kTrSearchL1, 1);
    pdl_trigger_search();
    // thread 0: stage the operands of sub-FFT (tn, k2n) -- E always, D (into S1 half `half`) only while the capture is new
    auto issue = [&](const TileIdx &tn, bool fresh_n, int k2n, int half) {
        const int r = (k2n - tn.dop) & 3;
        const int q = (k2n - tn.dop - r) >> 2;
        const float2 *Ek = p.Ep + (size_t)(tn.sat * 4 + r) * p.ext_len + ((p.Q + q) & ~1);
        fence_proxy_async();  // generic-proxy reads of these buffers (ordered by the CTA barrier) before the async writes
        mbar_expect_tx(bar, (uint32_t)(sizeof(float2) * (kEBufElems + (fresh_n ? kSub : 0))));
        tma_load_1d(smem_u32(s.E), Ek, (uint32_t)(sizeof(float2) * kEBufElems), bar);
        if (fresh_n) {
            const float2 *Dk = p.Dp + d_row(p, tn, 0) * kN + k2n * kSub;
            tma_load_1d(smem_u32(s.S1 + half * kSub), Dk, (uint32_t)(sizeof(float2) * kSub), bar);
        }
    };
    // Chunk feed.  The CTA's first chunk is number blockIdx.x (the grid never exceeds the chunk count); thread 0 claims
    // the next one during the first sub-FFT of a chunk's LAST tile, publishes the next tile (inside the chunk: the
    // successor) behind the barrier of sub-FFT 2 and stages it behind that of sub-FFT 3.  feed[8]: the next tile belongs
    // to another capture (D is staged and parked again), feed[9]: tiles left in its chunk behind it.
    int *feed = red_i + 20;
    unsigned cur, left;
    chunk_of(p, blockIdx.x, cur, left);
    left -= 1;
    TileIdx ti(p, cur);
    bool fresh = true;
    unsigned nxt_chunk = blockIdx.x;   // thread 0: the chunk being run, then the claimed one
    if (t == 0) issue(ti, true, 0, 0);
    int it = 0;  // sub-FFT counter: S1 half and mbarrier phase parity = it & 1
    int par = 0, pend_cap = -1, pend_slot = 0, pend_d = 0;
    auto flush = [&]() {   // thread 0: the previous tile's peak (deferred cross-warp merge, see k_search_l1)
        store_cell(p, pend_cap, pend_slot, pend_d, merge_warp_peaks(red_f + 16 * (par ^ 1), red_i + 8 * (par ^ 1)), L);
    };

    for (;;) {
        float P[16];
        float2 acc[16];
        float2 x[16];
        // aided: by two (at four the window base in thread 0's publish_tile costs the loop a 28-byte spill)
        constexpr int kCrUnroll = PA::kAided ? 2 : ACQ_CR_UNROLL;
#pragma unroll kCrUnroll
        for (int k2 = 0; k2 < 4; k2++) {
            float2 *S1b = s.S1 + (it & 1) * kSub;
            const int r = (k2 - ti.dop) & 3;
            const int q = (k2 - ti.dop - r) >> 2;
            const float2 *Ek = s.E + ((p.Q + q) & 1) + t;
            if (fresh) {   // D from the staged residue; park this thread's 16 values for the capture's other tiles
                const float2 *Dk = S1b + t;
                mbar_wait(bar, (uint32_t)(it & 1));
#pragma unroll
                for (int a = 0; a < 16; a++) x[a] = Dk[256 * a];
                tmem_st16(d_taddr + 32 * k2, x);
                tmem_wait_st();
            } else {
                tmem_ld16(d_taddr + 32 * k2, x);
                mbar_wait(bar, (uint32_t)(it & 1));
                tmem_wait_ld();
            }
            // x[a] = conj(data[k]) * code[k - dop], k = 1024 a + 4 t + k2   (search.cpp:471)
#pragma unroll
            for (int a = 0; a < 16; a++) x[a] = cmul_conj_a(x[a], Ek[256 * a]);
            subfft4096_inv4s(x, k2, bw, S1b, t, s.T2, BaseFromGlobal{bases}, [&]() {
                if (t == 0) {  // every warp is past its operand reads of this sub-FFT and past stage C of the previous one
                    if (k2 == 0 && left == 0) nxt_chunk = p.tile_ctr ? gridDim.x + atomicAdd(p.tile_ctr, 1u) : nxt_chunk + gridDim.x;
                    if (k2 == 2) {
                        unsigned ntile = cur + 1, nleft = left - 1;
                        bool valid = true;
                        if (left == 0) {
                            valid = chunk_of(p, nxt_chunk, ntile, nleft);
                            nleft -= 1;
                        }
                        publish_tile(feed, p, valid ? ntile : kNoTile);
                        feed[8] = valid && feed[3] != ti.cap;
                        feed[9] = (int)nleft;
                        feed[10] = (int)ntile;
                    }
                    if (k2 < 3) issue(ti, fresh, k2 + 1, (it + 1) & 1);
                    else {
                        TileIdx tn;
                        if (next_tile(feed, tn)) issue(tn, feed[8] != 0, 0, (it + 1) & 1);
                    }
                }
            });
            it++;
            if (t == 0 && k2 == 0 && pend_cap >= 0) flush();
            if (k2 == 0) {
#pragma unroll
                for (int n2 = 0; n2 < 16; n2++) acc[n2] = x[r16(n2)];
            } else {
#pragma unroll
                for (int n2 = 0; n2 < 16; n2++) acc[n2] = cfma(x[r16(n2)], c_cC[k2][n2], acc[n2]);
            }
        }
#pragma unroll
        for (int n2 = 0; n2 < 16; n2++) P[n2] = cpower(acc[n2]);
        warp_reduce_peak_redux(thread_peak_l1(P, t), red_f + 16 * par, red_i + 8 * par, t);
        pend_cap = ti.cap;
        pend_slot = ti.slot;
        pend_d = ti.d;
        par ^= 1;
        if (!next_tile(feed, ti)) break;   // published behind the barrier of sub-FFT 2, read behind that of sub-FFT 3
        fresh = feed[8] != 0;
        left = (unsigned)feed[9];
        cur = (unsigned)feed[10];
    }
    __syncthreads();
    if (t == 0 && pend_cap >= 0) flush();
    claims_done(p, t);
    search_cta_epilogue(p, t);
    ACQ_TRACE_STAMP(kTrSearchL1, 2);
    tmem_free_cta<2 * kTwCols>(tmem_base, t);
}

// Tensor memory (TMEM, 256 KB per SM) as thread-private scratch.  The E1B combine needs the outputs of three
// residues parked while the fourth is computed: 48 complex values per thread, 96 KiB per CTA.  In shared memory
// that scratch limits the kernel to one CTA per SM and puts 96 extra loads/stores per thread and tile on the
// L1/shared data pipe, the kernel's busiest unit.  TMEM is exactly "512 columns of 32 bits per thread lane":
// tcgen05.st / tcgen05.ld (.32x32b: thread i of the warp <-> lane 32*(warp%4)+i, N consecutive columns <-> N
// registers) move the parked values over the tensor-memory datapath instead.  Warps w and w+4 share lanes and
// use disjoint column ranges; a CTA allocates 256 columns, so two CTAs fill the SM's 512.
constexpr int kE1bTmemCols = 256;  // 2 warp sets x 96 columns, rounded up to a power of two

// k_search_e1b: as k_search_e1b_ldg, with the operand staging of k_search_l1 -- both operands of a sub-FFT land in
// shared memory by TMA bulk copies issued one sub-FFT ahead (D into the idle half of the exchange buffer, E into
// its own buffer), the B->C tiles live inside the exchange rows, and the cross-warp peak merge is deferred to the
// next tile (no reduction barrier).  A thread's 128 TMEM columns hold the three parked residues (96) and the four
// stage-A bases (8), so the stage-B twiddles stay in a 7.5 KiB shared-memory table.  106 KiB of shared memory per
// CTA, two CTAs per SM.
#ifndef ACQ_E1B_BEST4
#define ACQ_E1B_BEST4 1
#endif
constexpr int kE1bBaseCol = 96;  // TMEM columns [96, 104): W16384^{4t+k2}, k2 = 0..3
// Unroll factor of the residue loop (see ACQ_K2_UNROLL): measured on cfg3 19.6 M tiles/s rolled, 19.9 M by two,
// 20.4 M fully unrolled (the park/no-park branch and the residue-dependent constants fold away; 24 bytes of spill).
#ifndef ACQ_E1B_K2_UNROLL
#define ACQ_E1B_K2_UNROLL 4
#endif
constexpr int kE1bK2Unroll = ACQ_E1B_K2_UNROLL;
struct E1bSmem {
    float2 *S1;  // [2][4096]
    float2 *E;   // [4098]
    unsigned long long *bar;
    float2 *T2;  // [4][15][16]
    float *red_f;
    int *red_i;
};
__host__ __device__ constexpr size_t e1b_smem_bytes()
{
    return sizeof(float2) * (size_t)(2 * kSub + kEBufElems) + 16 + sizeof(float2) * kT2Elems + 64 * sizeof(float);
}
__device__ __forceinline__ E1bSmem e1b_smem_carve(unsigned char *base)
{
    E1bSmem s;
    s.S1 = reinterpret_cast<float2 *>(base);
    s.E = s.S1 + 2 * kSub;
    s.bar = reinterpret_cast<unsigned long long *>(s.E + kEBufElems);
    s.T2 = reinterpret_cast<float2 *>(s.bar + 2);
    s.red_f = reinterpret_cast<float *>(s.T2 + kT2Elems);  // [2 parities][16], then the TMEM slot at [48]
    s.red_i = reinterpret_cast<int *>(s.red_f + 32);        // [2 parities][8]
    return s;
}

template <class PA>
__global__ void __launch_bounds__(256, 2) k_search_e1b(const PA p)
{
    extern __shared__ __align__(1024) unsigned char smem[];
    const E1bSmem s = e1b_smem_carve(smem);
    float *red_f = s.red_f;
    int *red_i = s.red_i;
    const int t = threadIdx.x;
    constexpr int L = ACQ_LAGS_E1B;
    ACQ_TRACE_STAMP(kTrSearchE1b, 0);
    const uint32_t tmem_base = tmem_alloc_cta<kE1bTmemCols>(reinterpret_cast<uint32_t *>(red_f + 48), t);
    {   // stage-B twiddle table into shared memory
        const float4 *src = reinterpret_cast<const float4 *>(p.tables);
        float4 *dst = reinterpret_cast<float4 *>(s.T2);
        for (int i = t; i < kT2Elems / 2; i += 256) dst[i] = __ldg(src + i);
    }
    // this thread's TMEM: lane 32*(warp%4) + (t%32), columns [128*(warp/4), +128): [k2][n2] parked, then the bases
    const uint32_t zaddr = tmem_base + tmem_lane_base(t) + (uint32_t)((t >> 7) * 128);
    float2 bw = __ldg(p.tables + kT2Elems + t);  // W16384^{4t}: base of residue 0
    tmem_st1(zaddr + kE1bBaseCol, bw);
#pragma unroll
    for (int k2 = 1; k2 < 4; k2++) tmem_st1(zaddr + kE1bBaseCol + 2 * k2, __ldg(p.tables + kT2Elems + k2 * 256 + t));
    tmem_wait_st();
    const uint32_t bar = smem_u32(s.bar);
    if (t == 0) mbar_init(bar, 1);
    __syncthreads();
    if (p.wait_prior) pdl_wait();
    ACQ_TRACE_STAMP(kTrSearchE1b, 1);
    pdl_trigger_search();
    auto issue = [&](const TileIdx &tn, int k2n, int half) {  // thread 0: stage the operands of sub-FFT (tn, k2n)
        const int r = (k2n - tn.dop) & 3;
        const int q = (k2n - tn.dop - r) >> 2;
        const float2 *Dk = p.Dp + d_row(p, tn, 0) * kN + k2n * kSub;
        const float2 *Ek = p.Ep + (size_t)(tn.sat * 4 + r) * p.ext_len + ((p.Q + q) & ~1);
        fence_proxy_async();  // generic-proxy reads of these buffers (ordered by the CTA barrier) before the async writes
        mbar_expect_tx(bar, (uint32_t)(sizeof(float2) * (kSub + kEBufElems)));
        tma_load_1d(smem_u32(s.E), Ek, (uint32_t)(sizeof(float2) * kEBufElems), bar);
        tma_load_1d(smem_u32(s.S1 + half * kSub), Dk, (uint32_t)(sizeof(float2) * kSub), bar);
    };
    TileIdx ti(p, blockIdx.x);   // the grid never exceeds the tile count: every CTA has a first tile
    if (t == 0) issue(ti, 0, 0);
    int *feed = red_i + 20;      // dynamic tile feed (claim_tile / publish_tile / next_tile)
    unsigned nxt = blockIdx.x;   // thread 0: the tile being run, then the claimed one
    int it = 0;  // sub-FFT counter: S1 half and mbarrier phase parity = it & 1
    int par = 0, pend_cap = -1, pend_slot = 0, pend_d = 0;
    auto flush = [&]() {   // thread 0: the previous tile's peak (deferred cross-warp merge)
        store_cell(p, pend_cap, pend_slot, pend_d, merge_warp_peaks(red_f + 16 * (par ^ 1), red_i + 8 * (par ^ 1)), L);
    };

    for (;;) {
        float2 x[16];
#pragma unroll kE1bK2Unroll
        for (int k2 = 0; k2 < 4; k2++) {
            float2 *S1b = s.S1 + (it & 1) * kSub;
            {   // x[a] = conj(data[k]) * code[k - dop], k = 1024 a + 4 t + k2   (search.cpp:471), operands from smem
                const int r = (k2 - ti.dop) & 3;
                const int q = (k2 - ti.dop - r) >> 2;
                const float2 *Dk = S1b + t;
                const float2 *Ek = s.E + ((p.Q + q) & 1) + t;
                mbar_wait(bar, (uint32_t)(it & 1));
#pragma unroll
                for (int a = 0; a < 16; a++) x[a] = cmul_conj_a(Dk[256 * a], Ek[256 * a]);
            }
            subfft4096_inv4s(x, k2, bw, S1b, t, s.T2, BaseFromTmem{zaddr + kE1bBaseCol}, [&]() {
                if (t == 0) {  // every warp is past its operand reads of this sub-FFT and past stage C of the previous one
                    if (k2 == 0) nxt = claim_tile(p, nxt);
                    if (k2 == 2) publish_tile(feed, p, nxt);
                    if (k2 < 3) issue(ti, k2 + 1, (it + 1) & 1);
                    else {
                        TileIdx tn;
                        if (next_tile(feed, tn)) issue(tn, 0, (it + 1) & 1);
                    }
                }
            });
            it++;
            if (t == 0 && k2 == 0 && pend_cap >= 0) flush();  // previous tile's peak
            if (k2 < 3) {
                float2 z[16];
#pragma unroll
                for (int n2 = 0; n2 < 16; n2++) z[n2] = (k2 == 0) ? x[r16(n2)] : cmul(x[r16(n2)], c_cC[k2][n2]);
                tmem_st16(zaddr + 32 * k2, z);
                tmem_wait_st();
            }
        }
        // radix-4 combine over k2, lags n = lag_of3(t, n2) + 4096 m < 16368.  Lags are not visited in
        // increasing order here, so ties compare the index explicitly (first index wins, search.cpp:488).
#if ACQ_E1B_BEST4
        // A thread's lags grow with n2 inside a quarter m and with m across quarters: one running (max, n2) per
        // quarter with a strict >, merged in the order m = 0..3 with a strict >, keeps the first maximum
        // (search.cpp:488) without comparing indices.
        float bp[4] = {0.0f, 0.0f, 0.0f, 0.0f}, bsum = 0.0f;
        int bn2[4] = {0, 0, 0, 0};
        const int lag0 = lag_of3(t, 0);
#pragma unroll
        for (int c4 = 0; c4 < 4; c4++) {
            float2 za[4], zb[4], zc[4];
            tmem_ld4(zaddr + 0 * 32 + 8 * c4, za);
            tmem_ld4(zaddr + 1 * 32 + 8 * c4, zb);
            tmem_ld4(zaddr + 2 * 32 + 8 * c4, zc);
            tmem_wait_ld();
#pragma unroll
            for (int i = 0; i < 4; i++) {
                const int n2 = 4 * c4 + i;
                float2 z0 = za[i], z1 = zb[i], z2 = zc[i];
                float2 z3 = cmul(x[r16(n2)], c_cC[3][n2]);
                radix4_inv(z0, z1, z2, z3);  // z_m = sum_k2 z_k2 * j^{k2*m}
                const float2 zz[4] = {z0, z1, z2, z3};
#pragma unroll
                for (int m = 0; m < 4; m++) {
                    const float pw = cpower(zz[m]);
                    // only the last 16 lags of the transform (m = 3, n2 = 15, t & 15 == 15) lie beyond L = 16368
                    if (m < 3 || n2 < 15 || lag0 + 256 * 15 + 4096 * 3 < L) {
                        if (pw > bp[m]) bp[m] = pw, bn2[m] = n2;
                        bsum += pw;
                    }
                }
            }
        }
        Peak best;
        best.p = 0.0f;
        best.n = 0x7fffffff;
        best.sum = bsum;
#pragma unroll
        for (int m = 0; m < 4; m++)
            if (bp[m] > best.p) best.p = bp[m], best.n = lag0 + 256 * bn2[m] + 4096 * m;
#else
        Peak best;
        best.p = 0.0f;
        best.n = 0x7fffffff;
        best.sum = 0.0f;
#pragma unroll
        for (int c4 = 0; c4 < 4; c4++) {
            float2 za[4], zb[4], zc[4];
            tmem_ld4(zaddr + 0 * 32 + 8 * c4, za);
            tmem_ld4(zaddr + 1 * 32 + 8 * c4, zb);
            tmem_ld4(zaddr + 2 * 32 + 8 * c4, zc);
            tmem_wait_ld();
#pragma unroll
            for (int i = 0; i < 4; i++) {
                const int n2 = 4 * c4 + i;
                float2 z0 = za[i], z1 = zb[i], z2 = zc[i];
                float2 z3 = cmul(x[r16(n2)], c_cC[3][n2]);
                radix4_inv(z0, z1, z2, z3);  // z_m = sum_k2 z_k2 * j^{k2*m}
                const float2 zz[4] = {z0, z1, z2, z3};
#pragma unroll
                for (int m = 0; m < 4; m++) {
                    const int n = lag_of3(t, n2) + 4096 * m;
                    const float pw = cpower(zz[m]);
                    if (n < L) peak_merge(best, pw, n, pw);
                }
            }
        }
#endif
        // parity slot `par` was last read (flush) during the previous tile, before >= 3 CTA barriers
        warp_reduce_peak(best, red_f + 16 * par, red_i + 8 * par, t);
        pend_cap = ti.cap;
        pend_slot = ti.slot;
        pend_d = ti.d;
        par ^= 1;
        if (!next_tile(feed, ti)) break;   // published behind the barrier of sub-FFT 2, read behind that of sub-FFT 3
    }
    __syncthreads();
    if (t == 0 && pend_cap >= 0) flush();
    claims_done(p, t);
    search_cta_epilogue(p, t);
    ACQ_TRACE_STAMP(kTrSearchE1b, 2);
    tmem_free_cta<kE1bTmemCols>(tmem_base, t);
}

// k_search_e1b_multi -- Galileo E1B with k_noncoh > 1 on ONE CTA per tile (two per SM), replacing the cluster form for
// non-coherent sums (which has 0.35x the throughput once there are more tiles than clusters).  A thread owns 64 lags
// (16 values of n2 x 4 quarters m) whose block powers must survive from block to block: 64 floats on top of the 96
// tensor-memory columns the three parked residues occupy.  They do not fit the thread's 128 columns, so the powers of
// n2 >= 8 live in the 32 columns that remain and those of n2 < 8 in a thread-private 32 KiB shared-memory array that
// takes the place of the code-run staging buffer; the code operand E comes straight from L2 instead (16 loads per
// thread and sub-FFT, issued before the wait for the capture residue D, which is still TMA-staged one sub-FFT ahead),
// and the stage-A bases from the 8 KiB global table.  Block b was delayed by 16 b samples in the front end, so lag n
// lines up across blocks exactly as in k_search_l1_multi.  Same 106 KiB of shared memory as k_search_e1b.
struct E1bMultiSmem {
    float2 *S1;  // [2][4096]
    float *Ps;   // [32][256] block powers of this thread's lags with n2 < 8: index 4 n2 + m
    unsigned long long *bar;
    float2 *T2;  // [4][15][16]
    float *red_f;
    int *red_i;
};
__host__ __device__ constexpr size_t e1b_multi_smem_bytes()
{
    return sizeof(float2) * (size_t)(2 * kSub) + sizeof(float) * 32 * 256 + 16 + sizeof(float2) * kT2Elems + 64 * sizeof(float);
}
constexpr int kE1bPowCol = 96;  // TMEM columns [96, 128): block powers of the lags with n2 >= 8, index 4 (n2 - 8) + m

// Residue loop fully unrolled (16 bytes of spill): cfg3 with K = 4 0.721 ms rolled, 0.716 by two, 0.701 by four.
#ifndef ACQ_E1B_MULTI_UNROLL
#define ACQ_E1B_MULTI_UNROLL 4
#endif
template <class PA>
__global__ void __launch_bounds__(256, 2) k_search_e1b_multi(const PA p)
{
    extern __shared__ __align__(1024) unsigned char smem[];
    E1bMultiSmem s;
    s.S1 = reinterpret_cast<float2 *>(smem);
    s.Ps = reinterpret_cast<float *>(s.S1 + 2 * kSub);
    s.bar = reinterpret_cast<unsigned long long *>(s.Ps + 32 * 256);
    s.T2 = reinterpret_cast<float2 *>(s.bar + 2);
    s.red_f = reinterpret_cast<float *>(s.T2 + kT2Elems);
    s.red_i = reinterpret_cast<int *>(s.red_f + 32);
    float *red_f = s.red_f;
    int *red_i = s.red_i;
    const int t = threadIdx.x;
    constexpr int L = ACQ_LAGS_E1B;
    ACQ_TRACE_STAMP(kTrSearchE1b, 0);
    const uint32_t tmem_base = tmem_alloc_cta<kE1bTmemCols>(reinterpret_cast<uint32_t *>(red_f + 48), t);
    {   // stage-B twiddle table into shared memory
        const float4 *src = reinterpret_cast<const float4 *>(p.tables);
        float4 *dst = reinterpret_cast<float4 *>(s.T2);
        for (int i = t; i < kT2Elems / 2; i += 256) dst[i] = __ldg(src + i);
    }
    const uint32_t zaddr = tmem_base + tmem_lane_base(t) + (uint32_t)((t >> 7) * 128);
    const float2 *bases = p.tables + kT2Elems + t;
    float2 bw = __ldg(bases);
    float *Pt = s.Ps + t;
    const uint32_t bar = smem_u32(s.bar);
    if (t == 0) mbar_init(bar, 1);
    __syncthreads();
    if (p.wait_prior) pdl_wait();
    ACQ_TRACE_STAMP(kTrSearchE1b, 1);
    pdl_trigger_search();
    auto issue = [&](const TileIdx &tn, int bn, int k2n, int half) {  // thread 0: stage the capture residue of sub-FFT (tn, bn, k2n)
        const float2 *Dk = p.Dp + d_row(p, tn, bn) * kN + k2n * kSub;
        fence_proxy_async();
        mbar_expect_tx(bar, (uint32_t)(sizeof(float2) * kSub));
        tma_load_1d(smem_u32(s.S1 + half * kSub), Dk, (uint32_t)(sizeof(float2) * kSub), bar);
    };
    TileIdx ti(p, blockIdx.x);   // the grid never exceeds the tile count: every CTA has a first tile
    if (t == 0) issue(ti, 0, 0, 0);
    int *feed = red_i + 20;      // dynamic tile feed (claim_tile / publish_tile / next_tile)
    unsigned nxt = blockIdx.x;   // thread 0: the tile being run, then the claimed one
    int it = 0;
    int par = 0, pend_cap = -1, pend_slot = 0, pend_d = 0;
    auto flush = [&]() {   // thread 0: the previous tile's peak (deferred cross-warp merge)
        store_cell(p, pend_cap, pend_slot, pend_d, merge_warp_peaks(red_f + 16 * (par ^ 1), red_i + 8 * (par ^ 1)), L);
    };
    const int lag0 = lag_of3(t, 0);

    for (;;) {
        float bp[4] = {0.0f, 0.0f, 0.0f, 0.0f}, bsum = 0.0f;   // last block: running maximum per quarter, sum
        int bn2[4] = {0, 0, 0, 0};
        for (int b = 0; b < p.K; b++) {
            float2 x[16];
            constexpr int kE1bMultiUnroll = ACQ_E1B_MULTI_UNROLL;
#pragma unroll kE1bMultiUnroll
            for (int k2 = 0; k2 < 4; k2++) {
                float2 *S1b = s.S1 + (it & 1) * kSub;
                {   // x[a] = conj(data[k]) * code[k - dop], k = 1024 a + 4 t + k2   (search.cpp:471); E straight from L2
                    const int r = (k2 - ti.dop) & 3;
                    const int q = (k2 - ti.dop - r) >> 2;
                    const float2 *Eg = p.Ep + (size_t)(ti.sat * 4 + r) * p.ext_len + p.Q + q + t;
                    const float2 *Dk = S1b + t;
#pragma unroll
                    for (int a = 0; a < 16; a++) x[a] = __ldg(Eg + 256 * a);
                    mbar_wait(bar, (uint32_t)(it & 1));
#pragma unroll
                    for (int a = 0; a < 16; a++) x[a] = cmul_conj_a(Dk[256 * a], x[a]);
                }
                subfft4096_inv4s(x, k2, bw, S1b, t, s.T2, BaseFromGlobal{bases}, [&]() {
                    if (t == 0) {
                        if (b == 0 && k2 == 0) nxt = claim_tile(p, nxt);
                        if (b == p.K - 1 && k2 == 2) publish_tile(feed, p, nxt);
                        if (k2 < 3) issue(ti, b, k2 + 1, (it + 1) & 1);
                        else if (b + 1 < p.K) issue(ti, b + 1, 0, (it + 1) & 1);
                        else {
                            TileIdx tn;
                            if (next_tile(feed, tn)) issue(tn, 0, 0, (it + 1) & 1);
                        }
                    }
                });
                it++;
                if (t == 0 && b == 0 && k2 == 0 && pend_cap >= 0) flush();  // previous tile's peak
                if (k2 < 3) {
                    float2 z[16];
#pragma unroll
                    for (int n2 = 0; n2 < 16; n2++) z[n2] = (k2 == 0) ? x[r16(n2)] : cmul(x[r16(n2)], c_cC[k2][n2]);
                    tmem_st16(zaddr + 32 * k2, z);
                    tmem_wait_st();
                }
            }
            // radix-4 combine over k2 for this block, power, accumulation over blocks; on the last block the peak
            const bool first = (b == 0), last = (b + 1 == p.K);
#pragma unroll
            for (int c4 = 0; c4 < 4; c4++) {
                float2 za[4], zb[4], zc[4];
                tmem_ld4(zaddr + 0 * 32 + 8 * c4, za);
                tmem_ld4(zaddr + 1 * 32 + 8 * c4, zb);
                tmem_ld4(zaddr + 2 * 32 + 8 * c4, zc);
                float2 ph[8];   // previous sums of this quarter's 16 lags (index 4 i + m), as pairs
                if (!first) {
                    if (c4 >= 2) tmem_ld8(zaddr + kE1bPowCol + 16 * (c4 - 2), ph);
                    else {
#pragma unroll
                        for (int j = 0; j < 8; j++) ph[j] = make_float2(Pt[(16 * c4 + 2 * j) * 256], Pt[(16 * c4 + 2 * j + 1) * 256]);
                    }
                }
                tmem_wait_ld();
                float pw[16];
#pragma unroll
                for (int i = 0; i < 4; i++) {
                    const int n2 = 4 * c4 + i;
                    float2 z0 = za[i], z1 = zb[i], z2 = zc[i];
                    float2 z3 = cmul(x[r16(n2)], c_cC[3][n2]);
                    radix4_inv(z0, z1, z2, z3);  // z_m = sum_k2 z_k2 * j^{k2*m}
                    const float2 zz[4] = {z0, z1, z2, z3};
#pragma unroll
                    for (int m = 0; m < 4; m++) {
                        const int idx = 4 * i + m;
                        const float prev = first ? 0.0f : ((idx & 1) ? ph[idx >> 1].y : ph[idx >> 1].x);
                        pw[idx] = first ? cpower(zz[m]) : prev + cpower(zz[m]);
                    }
                }
                if (!last) {
                    if (c4 >= 2) {
                        float2 ps[8];
#pragma unroll
                        for (int j = 0; j < 8; j++) ps[j] = make_float2(pw[2 * j], pw[2 * j + 1]);
                        tmem_st8(zaddr + kE1bPowCol + 16 * (c4 - 2), ps);
                        tmem_wait_st();
                    } else {
#pragma unroll
                        for (int j = 0; j < 16; j++) Pt[(16 * c4 + j) * 256] = pw[j];
                    }
                } else {
#pragma unroll
                    for (int i = 0; i < 4; i++) {
                        const int n2 = 4 * c4 + i;
#pragma unroll
                        for (int m = 0; m < 4; m++) {
                            // only the last 16 lags of the transform (m = 3, n2 = 15, t & 15 == 15) lie beyond L = 16368
                            if (m < 3 || n2 < 15 || lag0 + 256 * 15 + 4096 * 3 < L) {
                                if (pw[4 * i + m] > bp[m]) bp[m] = pw[4 * i + m], bn2[m] = n2;
                                bsum += pw[4 * i + m];
                            }
                        }
                    }
                }
            }
        }
        // a thread's lags grow with n2 inside a quarter and with m across quarters: strict > in that order keeps the
        // first maximum (search.cpp:488)
        Peak best;
        best.p = 0.0f;
        best.n = 0x7fffffff;
        best.sum = bsum;
#pragma unroll
        for (int m = 0; m < 4; m++)
            if (bp[m] > best.p) best.p = bp[m], best.n = lag0 + 256 * bn2[m] + 4096 * m;
        warp_reduce_peak(best, red_f + 16 * par, red_i + 8 * par, t);
        pend_cap = ti.cap;
        pend_slot = ti.slot;
        pend_d = ti.d;
        par ^= 1;
        if (!next_tile(feed, ti)) break;   // published behind the barrier of the second-to-last sub-FFT, read behind the last
    }
    __syncthreads();
    if (t == 0 && pend_cap >= 0) flush();
    claims_done(p, t);
    search_cta_epilogue(p, t);
    ACQ_TRACE_STAMP(kTrSearchE1b, 2);
    tmem_free_cta<kE1bTmemCols>(tmem_base, t);
}

// ---------------------------------------------------------------------------------------------
// K3-5, cluster form of the E1B search: one tile per thread-block CLUSTER of four CTAs.  CTA rank k2 runs the
// 4096-point sub-FFT of input residue k2 (all four in parallel on four SMs) and publishes its twiddled output
// Y_k2[n'] in its own shared memory.  After a cluster barrier CTA rank c forms ALL FOUR lag quarters for its
// slice of n' (n2 in 4c .. 4c+3),
//     r[n' + 4096 m] = sum_k2 j^{k2 m} Y_k2[n'],      m = 0..3,
// reading the other three CTAs' slices through distributed shared memory (DSMEM, ld.shared::cluster): 24 KiB of
// remote reads per CTA and tile.  (Splitting by m instead would make every CTA read all of every Y: 96 KiB.)
// Peaks are reduced per CTA, sent to rank 0 through DSMEM and merged there; only the 16-byte cell leaves the
// cluster.  No thread-private scratch, four SMs per tile: shorter latency per tile and a 4x finer scheduling
// grain than k_search_e1b.  The host picks the form in acq_api.cu (ACQ_E1B_KERNEL=cta|cluster forces one).
// MULTI (k_noncoh > 1): each thread owns 16 lags (4 values of n2 x 4 quarters), so the block powers are summed
// in registers exactly as in k_search_l1 (front-end block delay, see k_hb2).  Y is double
// buffered: one cluster barrier per block (a buffer is rewritten two blocks later, after the barrier every
// CTA reached only when it had finished reading it).
template <bool MULTI, class PA>
__global__ void __cluster_dims__(4, 1, 1) __launch_bounds__(256, 1) k_search_e1b_cluster(const PA p)
{
    namespace cg = cooperative_groups;
    cg::cluster_group cluster = cg::this_cluster();
    extern __shared__ __align__(1024) unsigned char smem[];
    const FftSmem3 s = fft_smem3_carve(smem);
    float2 *Y = reinterpret_cast<float2 *>(smem + fft_smem3_bytes());            // [2][16][256] own residue
    float *red_f = reinterpret_cast<float *>(smem + fft_smem3_bytes() + 2 * sizeof(float2) * kSub);
    int *red_i = reinterpret_cast<int *>(red_f + 16);
    float *peaks_f = red_f + 32;  // [4][2] (peak, sum) per rank, filled through DSMEM in rank 0
    int *peaks_i = reinterpret_cast<int *>(red_f + 40);
    const int t = threadIdx.x;
    const int rank = (int)cluster.block_rank();  // = k2 in the sub-FFT phase, = n2 slice in the combine phase
    constexpr int L = ACQ_LAGS_E1B;
    load_t2(s, p.tables, t);
    const float2 bw = __ldg(p.tables + kT2Elems + rank * 256 + t);
    const float2 *Yr[4];
#pragma unroll
    for (int k = 0; k < 4; k++) Yr[k] = cluster.map_shared_rank(Y, k);
    float *peaks_f0 = cluster.map_shared_rank(peaks_f, 0);
    int *peaks_i0 = cluster.map_shared_rank(peaks_i, 0);
    const int n_clusters = gridDim.x >> 2;
    int buf = 0, yb = 0;
    if (p.wait_prior) pdl_wait();
    ACQ_TRACE_STAMP(kTrE1bCluster, 1);
    pdl_trigger_search();

    for (long long tile = blockIdx.x >> 2; tile < p.n_tiles; tile += n_clusters) {
        const TileIdx ti(p, tile);
        float P[16];
        for (int b = 0; b < p.K; b++) {
            float2 x[16];
            load_products(x, p, ti, b, rank, t);
            subfft4096_inv3(x, rank, bw, buf, s, t);
            buf ^= 1;
            float2 *Yw = Y + yb * kSub;
#pragma unroll
            for (int n2 = 0; n2 < 16; n2++)
                Yw[n2 * 256 + t] = (rank == 0) ? x[r16(n2)] : cmul(x[r16(n2)], c_cC[rank][n2]);
            cluster.sync();  // every Y_k2 of this block is complete and visible cluster-wide
#pragma unroll
            for (int i = 0; i < 4; i++) {
                const int o = yb * kSub + (4 * rank + i) * 256 + t;
                float2 z0 = Yr[0][o], z1 = Yr[1][o], z2 = Yr[2][o], z3 = Yr[3][o];
                radix4_inv(z0, z1, z2, z3);  // z_m = sum_k2 z_k2 * j^{k2*m}
                const float2 zz[4] = {z0, z1, z2, z3};
#pragma unroll
                for (int m = 0; m < 4; m++) {
                    const float pw = cpower(zz[m]);
                    P[4 * m + i] = (!MULTI || b == 0) ? pw : P[4 * m + i] + pw;
                }
            }
            yb ^= 1;
        }
        Peak best;
        best.p = 0.0f;
        best.n = 0x7fffffff;
        best.sum = 0.0f;
#pragma unroll
        for (int q = 0; q < 16; q++) {   // q = 4 m + i: this thread's lags in increasing order
            const int n = lag_of3(t, 4 * rank + (q & 3)) + 4096 * (q >> 2);
            if (n < L) {   // strict > keeps the first maximum (search.cpp:488)
                if (P[q] > best.p) best.p = P[q], best.n = n;
                best.sum += P[q];
            }
        }
        const Peak tot = block_reduce_peak(best, red_f, red_i, t);
        if (t == 0) {
            peaks_f0[2 * rank] = tot.p;
            peaks_f0[2 * rank + 1] = tot.sum;
            peaks_i0[rank] = tot.n;
        }
        cluster.sync();  // peaks have landed in rank 0
        if (rank == 0 && t == 0) {
            Peak all;
            all.p = peaks_f[0];
            all.sum = peaks_f[1];
            all.n = peaks_i[0];
#pragma unroll
            for (int k = 1; k < 4; k++) peak_merge(all, peaks_f[2 * k], peaks_i[k], peaks_f[2 * k + 1]);
            store_cell(p, ti.cap, ti.slot, ti.d, all, L);
        }
        // the peak slots are rewritten only after the next tile's first cluster barrier, which rank 0's
        // thread 0 reaches after the merge above
    }
    if (rank == 0) search_cta_epilogue(p, t);  // rank 0 stored the cluster's cells
}

// K5b for small searches (up to a few hundred rows): ONE CTA, chained to the search launches by programmatic dependent
// launch.  It does not wait for the search grids to complete (griddepcontrol.wait: grid drain + memory flush); thread 0
// polls the counter the search CTAs bump after their last cell (search_cta_epilogue), so the pick starts a fence and an
// atomic after the last cell is stored -- and C/A and E1B launches of one search need no ordering between them.
// Then 32 warps pick the rows, the counter is zeroed for the next search and, for a host that polls mapped memory,
// the completion word is raised behind the records.
__global__ void __launch_bounds__(1024) k_pick_small(const acq_cell *cells, const int *__restrict__ slot_sat, acq_record *out,
                                                    unsigned *ctas_done, unsigned ctas_total, unsigned *host_flag, unsigned epoch,
                                                    int n_rows, int n_slots, int n_dop, PickDop pd)
{
    // Records are staged in shared memory and leave in 16-byte pieces: written one 4-byte member at a time straight into
    // mapped host memory they cost 0.17 us per record (every store its own PCIe write: 6.8 us of a 74 us cold-start
    // search, 14 us for the 82 rows of the all-constellation search -- measured with the trace variant).  For a polling
    // host every 16-byte piece carries the epoch (acq_record_tagged): the 2..3.5 us of system fence + completion word
    // that used to close the kernel are gone.
    __shared__ __align__(16) acq_record s_rec[kPickSmallRowsMax];
    const int t = threadIdx.x;
    ACQ_TRACE_STAMP(kTrPick, 0);
    __shared__ unsigned s_timed_out;
    if (t == 0) {
        // Poll, but never hang the GPU: if the count does not arrive within 2 s (a search kernel that failed to run, a
        // count left over by an aborted search) the pick goes ahead on what is there and announces the failure
        // instead of the epoch; the counter is reset either way.
        const volatile unsigned *done = ctas_done;
        unsigned long long t0, now;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
        unsigned spins = 0;
        s_timed_out = 0;
        while (*done != ctas_total) {
            if ((++spins & 0x3fff) == 0) {
                asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
                if (now - t0 > 2000000000ull) {
                    s_timed_out = 1;
                    break;
                }
            }
        }
        __threadfence();
    }
    __syncthreads();
    ACQ_TRACE_STAMP(kTrPick, 1);
    pick_rows<4>(cells, slot_sat, s_rec, t >> 5, 32, n_rows, n_slots, n_dop, pd, t & 31);
    __syncthreads();
    ACQ_TRACE_STAMP(kTrPick, 3);
    if (host_flag) {
        // polled host: tagged 32-byte records, two 16-byte stores each (see acq_record_tagged); nothing to fence
        uint4 *dst = reinterpret_cast<uint4 *>(out);
        const unsigned tag = s_timed_out ? 0xffffffffu : epoch;   // a pick that gave up never announces records
        for (int i = t; i < n_rows; i += 1024) {
            const acq_record r = s_rec[i];
            dst[2 * i] = make_uint4((unsigned)r.sat, (unsigned)r.lag, (unsigned)r.dop, tag);
            dst[2 * i + 1] = make_uint4(__float_as_uint(r.peak), __float_as_uint(r.noise), __float_as_uint(r.snr), tag);
        }
        if (t == 0) {
            *ctas_done = 0;
            if (s_timed_out) *reinterpret_cast<volatile unsigned *>(host_flag) = 0xffffffffu;
        }
    } else {
        const int n16 = n_rows * (int)sizeof(acq_record) / 16;  // 24-byte records: an even row count is a whole number of pieces
        const uint4 *src = reinterpret_cast<const uint4 *>(s_rec);
        if ((reinterpret_cast<uintptr_t>(out) & 15) == 0) {
            uint4 *dst = reinterpret_cast<uint4 *>(out);
            for (int i = t; i < n16; i += 1024) dst[i] = src[i];
            const int tail = n16 * 16;  // odd row count: the last 8 bytes
            if (t == 0 && tail < n_rows * (int)sizeof(acq_record))
                *reinterpret_cast<uint2 *>(reinterpret_cast<char *>(out) + tail) =
                    *reinterpret_cast<const uint2 *>(reinterpret_cast<const char *>(s_rec) + tail);
        } else {
            for (int i = t; i < n_rows; i += 1024) out[i] = s_rec[i];
        }
        if (t == 0) *ctas_done = 0;
    }
    ACQ_TRACE_STAMP(kTrPick, 2);
}

// K5b for large searches: one warp per (capture, sat) row, after the search grids have completed.
__global__ void __launch_bounds__(128) k_best_dop(const acq_cell *__restrict__ cells, const int *__restrict__ slot_sat,
                                                  acq_record *__restrict__ out, int n_rows, int n_slots, int n_dop,
                                                  PickDop pd)
{
    pdl_wait();  // before the early exit: completion of this grid must imply completion of its predecessors
    ACQ_TRACE_STAMP(kTrPick, 1);
    pick_rows<1>(cells, slot_sat, out, blockIdx.x * 4 + (threadIdx.x >> 5), n_rows, n_rows, n_slots, n_dop, pd,
                 threadIdx.x & 31);
}

#if defined(ACQ_VARIANT_L1_LDG) || defined(ACQ_VARIANT_L1_X3) || defined(ACQ_VARIANT_E1B_LDG) || defined(ACQ_VARIANT_L1_SP) || \
    defined(ACQ_VARIANT_L1_ST) || defined(ACQ_VARIANT_L1_MST)
#include "acq_variants.cuh"  // A/B forms: experiment builds only (tools/build_variants.py)
#endif

// ---------------------------------------------------------------------------------------------
// K6.  Acquisition refinement for the hand-off to tracking (SURVEY 8(f) rank 4).  The search reports the code phase
// in /DECIM samples and the Doppler in bins of 249.76 Hz (search.cpp:574-575); the tracking loops then need a 5 s
// settle to pull in the LO (gps/channel.cpp:345-372) because +-125 Hz exceeds the Costas pull-in range.  For each
// record this kernel evaluates the correlation r_d[n] = sum_k conj(D[k]) C[k-d] e^{+j 2 pi k n / N} (the very sum
// the inverse FFT computes, search.cpp:471-481) at five points around the peak -- (d-1, n) (d, n-1) (d, n)
// (d, n+1) (d+1, n) -- straight from the spectra the search left in HBM, and forms
//   Doppler: delta = Re[(Xm - Xp) conj(2 X0 - Xm - Xp)] / |2 X0 - Xm - Xp|^2   (three-bin interpolation of a
//            rectangular-window DFT; X_d = r_d[n] e^{-j 2 pi d n / N} puts the three bins on a common phase),
//   code   : eps = slope (l - e) / (l + e),  e/l = Re(r[n-+1] conj(r[n]))       (early-minus-late over the
//            correlation triangle: 4 samples per chip -> slope 3; BOC(1,1) main peak -> slope 1/3),
// each summed over the K blocks.  One CTA per record; thread t owns k1 = t + 256 i for all four residues.
// ---------------------------------------------------------------------------------------------
struct RefineArgs {
    const float2 *Dp;
    const float2 *Ep;
    const acq_record *rec;   // [n_rows], row = cap * n_slots + slot
    const int *sat_type;     // [n_sats]
    acq_fine *out;
    int n_slots, K, nvar, half_bin, ext_len, Q, n_shift, smax, cd_div;
};

__global__ void __launch_bounds__(256) k_refine(const RefineArgs p)
{
    __shared__ float red[8][10];
    const int row = blockIdx.x, t = threadIdx.x;
    const acq_record rc = p.rec[row];
    const int cap = row / p.n_slots;
    const bool e1b = p.sat_type[rc.sat] == ACQ_E1B;
    const int v = p.half_bin ? (rc.dop & 1) : 0;
    const int dop = p.half_bin ? ((rc.dop - v) >> 1) : rc.dop;
    const int n = rc.lag;
    float num = 0.0f, den = 0.0f, early = 0.0f, late = 0.0f, peak = 0.0f;  // thread 0 only
    for (int b = 0; b < p.K; b++) {
        // the copy of block b the search read at this record's Doppler index (code-Doppler compensation), delayed
        // by 16 b + cshift samples in the front end
        const int cshift = p.n_shift > 1 ? code_shift(b, rc.dop, p.cd_div) : 0;
        const float2 *D = p.Dp + (((size_t)((size_t)cap * p.K + b) * p.nvar + v) * p.n_shift + (p.smax + cshift)) * kN;
        float2 acc[5];
#pragma unroll
        for (int j = 0; j < 5; j++) acc[j] = make_float2(0.0f, 0.0f);
        for (int k2 = 0; k2 < 4; k2++) {
            const float2 *Er[3];
#pragma unroll
            for (int j = 0; j < 3; j++) {  // code rows for Doppler dop-1, dop, dop+1
                const int dd = dop - 1 + j;
                const int r = (k2 - dd) & 3;
                const int q = (k2 - dd - r) >> 2;
                Er[j] = p.Ep + (size_t)(rc.sat * 4 + r) * p.ext_len + p.Q + q;
            }
            for (int k1 = t; k1 < kSub; k1 += 256) {
                const int k = 4 * k1 + k2;
                const float2 d = D[k2 * kSub + k1];
                float sn, cs, s1, c1;
                sincospif((float)((k * n) & (kN - 1)) * (1.0f / 8192.0f), &sn, &cs);  // e^{+j 2 pi k n / N}
                sincospif((float)k * (1.0f / 8192.0f), &s1, &c1);                      // e^{+j 2 pi k / N}
                const float2 w0 = make_float2(cs, sn), wk = make_float2(c1, s1);
                const float2 pm = cmul(cmul_conj_a(d, Er[0][k1]), w0);
                const float2 pc = cmul(cmul_conj_a(d, Er[1][k1]), w0);
                const float2 pp = cmul(cmul_conj_a(d, Er[2][k1]), w0);
                acc[0] = cadd(acc[0], pm);
                acc[1] = cadd(acc[1], cmul(pc, make_float2(c1, -s1)));  // lag n-1
                acc[2] = cadd(acc[2], pc);
                acc[3] = cadd(acc[3], cmul(pc, wk));                    // lag n+1
                acc[4] = cadd(acc[4], pp);
            }
        }
        // CTA reduction of the five complex sums
#pragma unroll
        for (int j = 0; j < 5; j++) {
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) {
                acc[j].x += __shfl_xor_sync(0xffffffffu, acc[j].x, off);
                acc[j].y += __shfl_xor_sync(0xffffffffu, acc[j].y, off);
            }
        }
        __syncthreads();  // red[] of the previous block has been consumed
        if ((t & 31) == 0) {
#pragma unroll
            for (int j = 0; j < 5; j++) {
                red[t >> 5][2 * j] = acc[j].x;
                red[t >> 5][2 * j + 1] = acc[j].y;
            }
        }
        __syncthreads();
        if (t == 0) {
            float2 R[5];
#pragma unroll
            for (int j = 0; j < 5; j++) {
                R[j] = make_float2(0.0f, 0.0f);
                for (int w = 0; w < 8; w++) R[j].x += red[w][2 * j], R[j].y += red[w][2 * j + 1];
            }
            float sn, cs;
            // w1 = e^{+j 2 pi n_b / N}, n_b = n + 16 b: the front end delayed block b by 16 b samples, so lag n of
            // its spectrum is lag n + 16 b of the block itself -- the lag the Doppler phase term refers to
            sincospif((float)((n + 16 * b + cshift) & (kN - 1)) * (1.0f / 8192.0f), &sn, &cs);
            const float2 Xm = cmul(R[0], make_float2(cs, sn)), Xp = cmul(R[4], make_float2(cs, -sn)), X0 = R[2];
            const float2 a = csub(Xm, Xp);
            const float2 g = csub(csub(cadd(X0, X0), Xm), Xp);
            num += a.x * g.x + a.y * g.y;
            den += g.x * g.x + g.y * g.y;
            early += R[1].x * R[2].x + R[1].y * R[2].y;
            late += R[3].x * R[2].x + R[3].y * R[2].y;
            peak += R[2].x * R[2].x + R[2].y * R[2].y;
        }
    }
    if (t == 0) {
        float delta = den > 0.0f ? num / den : 0.0f;
        delta = fminf(1.0f, fmaxf(-1.0f, delta));
        float eps = (early + late) > 0.0f ? (e1b ? (1.0f / 3.0f) : 3.0f) * (late - early) / (early + late) : 0.0f;
        eps = fminf(1.0f, fmaxf(-1.0f, eps));
        const int L = e1b ? ACQ_LAGS_E1B : ACQ_LAGS_L1;
        acq_fine o;
        o.dop_hz = ((p.half_bin ? 0.5f * (float)rc.dop : (float)rc.dop) + delta) * (float)ACQ_BIN_HZ;
        o.code_fs = (float)ACQ_DECIM * ((float)n + eps);
        o.peak = peak;
        int cs = (int)lrintf(o.code_fs) % (L * ACQ_DECIM);
        if (cs < 0) cs += L * ACQ_DECIM;
        o.ca_shift = cs;
        p.out[row] = o;
    }
}

// ---------------------------------------------------------------------------------------------
// launchers
// ---------------------------------------------------------------------------------------------
// Launch with (pdl) or without programmatic stream serialization: with it the grid may become resident while the
// preceding kernel of the stream is still running; its threads block in pdl_wait() until that kernel has completed.
template <class... KArgs, class... Args>
static void launch_k(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, bool pdl, Args... args)
{
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at;
    cfg.numAttrs = pdl ? 1 : 0;
    cudaLaunchKernelEx(&cfg, kern, KArgs(args)...);  // errors surface through cudaGetLastError() in the caller
}

static size_t search_l1_smem_bytes() { return fft_smem4_bytes() + 64 * sizeof(float); }
static size_t search_e1b_smem_bytes() { return e1b_smem_bytes(); }
static size_t search_e1b_cluster_smem_bytes() { return fft_smem3_bytes() + 2 * sizeof(float2) * kSub + 64 * sizeof(float); }
static size_t fwd_smem_bytes() { return fft_smem3_bytes() + kZBytes; }

#ifndef ACQ_CARVEOUT_MAX
#define ACQ_CARVEOUT_MAX 1   // 0 (variant carve0): the driver's choice per kernel
#endif

// The search kernels of an aided search (AidedSearchArgs): the product forms only, with the shared-memory size and carveout
// of their full-range instantiations.
static cudaError_t aided_kernels_configure()
{
    using A = AidedSearchArgs;
    const void *k[] = {(const void *)k_search_l1<false, A>, (const void *)k_search_l1_multi<A>, (const void *)k_search_l1_cr<A>,
                       (const void *)k_search_e1b<A>, (const void *)k_search_e1b_multi<A>, (const void *)k_search_e1b_cluster<false, A>,
                       (const void *)k_search_e1b_cluster<true, A>};
    const int smem[] = {(int)search_l1_smem_bytes(), (int)l1_multi_smem_bytes(), (int)l1_multi_smem_bytes(), (int)search_e1b_smem_bytes(),
                        (int)e1b_multi_smem_bytes(), (int)search_e1b_cluster_smem_bytes(), (int)search_e1b_cluster_smem_bytes()};
    cudaError_t e;
    for (int i = 0; i < 7; i++) {
        if ((e = cudaFuncSetAttribute(k[i], cudaFuncAttributeMaxDynamicSharedMemorySize, smem[i]))) return e;
#if ACQ_CARVEOUT_MAX
        if ((e = cudaFuncSetAttribute(k[i], cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared))) return e;
#endif
    }
    return cudaSuccess;
}

cudaError_t search_kernels_configure()
{
    using S = SearchArgs;
    cudaError_t e;
    const int l1 = (int)search_l1_smem_bytes(), e1 = (int)search_e1b_smem_bytes(), fw = (int)fwd_smem_bytes();
    if ((e = cudaFuncSetAttribute(k_search_l1<false, S>, cudaFuncAttributeMaxDynamicSharedMemorySize, l1))) return e;
#if ACQ_DR_MIN_TILES_PER_SM >= 0
    if ((e = cudaFuncSetAttribute(k_search_l1_dr, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dr_smem_bytes()))) return e;
#endif
#ifdef ACQ_VARIANT_L1_MST
    if ((e = cudaFuncSetAttribute(k_search_l1_mst, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dr_smem_bytes()))) return e;
#endif
#ifdef ACQ_VARIANT_L1_SP
    if ((e = cudaFuncSetAttribute(k_search_l1_sp, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sp_smem_bytes()))) return e;
#endif
#ifdef ACQ_VARIANT_L1_ST
    if ((e = cudaFuncSetAttribute(k_search_l1_st, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)st_smem_bytes()))) return e;
#endif
#ifdef ACQ_VARIANT_L1_MULTI_TW
    if ((e = cudaFuncSetAttribute(k_search_l1<true, S>, cudaFuncAttributeMaxDynamicSharedMemorySize, l1))) return e;
#endif
    if ((e = cudaFuncSetAttribute(k_search_l1_multi<S>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)l1_multi_smem_bytes()))) return e;
    if ((e = cudaFuncSetAttribute(k_search_l1_cr<S>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)l1_multi_smem_bytes()))) return e;
    if ((e = cudaFuncSetAttribute(k_search_e1b<S>, cudaFuncAttributeMaxDynamicSharedMemorySize, e1))) return e;
    if ((e = cudaFuncSetAttribute(k_search_e1b_multi<S>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)e1b_multi_smem_bytes()))) return e;
#ifdef ACQ_VARIANT_L1_X3
    const int l1x = (int)search_l1_x3_smem();
    if ((e = cudaFuncSetAttribute(k_search_l1_x3<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, l1x))) return e;
    if ((e = cudaFuncSetAttribute(k_search_l1_x3<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, l1x))) return e;
#endif
#ifdef ACQ_VARIANT_L1_LDG
    const int l1g = (int)(fft_smem3t_bytes() + 64 * sizeof(float));
    if ((e = cudaFuncSetAttribute(k_search_l1_ldg<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, l1g))) return e;
    if ((e = cudaFuncSetAttribute(k_search_l1_ldg<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, l1g))) return e;
#endif
#ifdef ACQ_VARIANT_E1B_LDG
    const int e1g = (int)(fft_smem3_bytes() + 64 * sizeof(float));
    if ((e = cudaFuncSetAttribute(k_search_e1b_ldg, cudaFuncAttributeMaxDynamicSharedMemorySize, e1g))) return e;
#endif
    const int ec = (int)search_e1b_cluster_smem_bytes();
    if ((e = cudaFuncSetAttribute(k_search_e1b_cluster<false, S>, cudaFuncAttributeMaxDynamicSharedMemorySize, ec))) return e;
    if ((e = cudaFuncSetAttribute(k_search_e1b_cluster<true, S>, cudaFuncAttributeMaxDynamicSharedMemorySize, ec))) return e;
    const int fc = (int)(fft_smem3_bytes() + 2 * sizeof(float2) * kSub);
    if ((e = cudaFuncSetAttribute(k_fwd_fft_cluster<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, fc))) return e;
    if ((e = cudaFuncSetAttribute(k_fwd_fft_cluster<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, fc))) return e;
    if ((e = cudaFuncSetAttribute(k_fwd_fft<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, fw))) return e;
    if ((e = cudaFuncSetAttribute(k_fwd_fft<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, fw))) return e;
    // One shared-memory carveout for every kernel of a search.  Left to the driver, the C/A kernel (2 x 96.3 KiB) runs
    // its SMs at the 196 KiB split and the E1B kernel (2 x 103.8 KiB) at 228 KiB, and an SM changes its split only when
    // it is empty: in a GPS + Galileo search the E1B CTAs -- launched to move in as the C/A CTAs retire -- entered no SM
    // before BOTH its C/A CTAs had gone (trace: first E1B CTA at 54.8 us although half the C/A CTAs leave by 50 us).
#if ACQ_CARVEOUT_MAX
    const void *chain[] = {(const void *)k_front_end<false>, (const void *)k_front_end<true>, (const void *)k_front_end_arg,
                           (const void *)k_fwd_fft<true>, (const void *)k_fwd_fft<false>, (const void *)k_fwd_fft_cluster<true>,
                           (const void *)k_fwd_fft_cluster<false>, (const void *)k_search_l1<false, S>,
#ifdef ACQ_VARIANT_L1_MULTI_TW
                           (const void *)k_search_l1<true, S>,
#endif
#if ACQ_DR_MIN_TILES_PER_SM >= 0
                           (const void *)k_search_l1_dr,
#endif
                           (const void *)k_search_l1_cr<S>, (const void *)k_search_l1_multi<S>, (const void *)k_search_e1b<S>,
                           (const void *)k_search_e1b_multi<S>, (const void *)k_search_e1b_cluster<false, S>,
                           (const void *)k_search_e1b_cluster<true, S>, (const void *)k_pick_small, (const void *)k_best_dop};
    for (const void *f : chain)
        if ((e = cudaFuncSetAttribute(f, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared))) return e;
#endif
    return aided_kernels_configure();
}

int launch_front_end(const uint8_t *packed, float2 *x2, const float2 *rot, int n_blocks, int nvar, int K, int sample_bits,
                     int n_shift, int smax, cudaStream_t st)
{
    int launched = 0;
    for (int b0 = 0; b0 < n_blocks; b0 += 32768) {  // gridDim.y <= 65535
        const int nb = (n_blocks - b0 < 32768) ? (n_blocks - b0) : 32768;
        const dim3 grid(kN / kFeOut, nb);
        if (sample_bits == 2)
            k_front_end<true><<<grid, 256, 0, st>>>(packed + (size_t)b0 * 2 * ACQ_BLOCK_BYTES,
                                                    x2 + (size_t)b0 * nvar * n_shift * kN, rot, nvar, K, b0, n_shift, smax);
        else
            k_front_end<false><<<grid, 256, 0, st>>>(packed + (size_t)b0 * ACQ_BLOCK_BYTES,
                                                     x2 + (size_t)b0 * nvar * n_shift * kN, rot, nvar, K, b0, n_shift, smax);
        launched++;
    }
    return launched;
}

// The same front end for ONE 1-bit block that still lies in host memory: the bytes travel as the kernel's argument.
int launch_front_end_arg(const uint8_t *packed_host, float2 *x2, const float2 *rot, int nvar, int n_shift, int smax,
                         cudaStream_t st)
{
    void *args[] = {const_cast<uint8_t *>(packed_host), &x2, &rot, &nvar, &n_shift, &smax};
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(kN / kFeOut, 1);
    cfg.blockDim = dim3(256);
    cfg.stream = st;
    if (cudaLaunchKernelExC(&cfg, reinterpret_cast<const void *>(k_front_end_arg), args) != cudaSuccess) return 0;
    return 1;
}

int launch_hb1_code(const uint32_t *chips, const int *codelen_boc, float2 *x1, int n_sats, cudaStream_t st)
{
    k_hb1_code<<<dim3(128, n_sats), 256, 0, st>>>(chips, codelen_boc, x1);
    return 1;
}

int launch_hb2(const float2 *x1, float2 *x2, const float2 *rot, int n_rows, int nvar, int K, cudaStream_t st)
{
    int launched = 0;
    for (int r0 = 0; r0 < n_rows; r0 += 32768) {
        const int nr = (n_rows - r0 < 32768) ? (n_rows - r0) : 32768;
        k_hb2<<<dim3(64, nr), 256, 0, st>>>(x1 + (size_t)r0 * 32768, x2 + (size_t)r0 * nvar * kN, rot, nvar, K, r0);
        launched++;
    }
    return launched;
}

int launch_fwd_fft(const float2 *x2, float2 *out, const float2 *tables, int n_rows, bool polyphase, int sm_count,
                   cudaStream_t st, bool pdl)
{
    if (n_rows <= sm_count / 4) {  // few rows: four CTAs per row (cluster + DSMEM), 2.5x shorter than the serial chain
        const size_t smem = fft_smem3_bytes() + 2 * sizeof(float2) * kSub;
        launch_k(polyphase ? k_fwd_fft_cluster<true> : k_fwd_fft_cluster<false>, 4 * n_rows, 256, smem, st, pdl, x2, out,
                 tables, n_rows);
        return 1;
    }
    const int grid = n_rows < sm_count ? n_rows : sm_count;
    launch_k(polyphase ? k_fwd_fft<true> : k_fwd_fft<false>, grid, 256, fwd_smem_bytes(), st, pdl, x2, out, tables, n_rows);
    return 1;
}

int launch_build_ext(const float2 *C, float2 *Ep, int n_sats, int Q, int ext_len, int wrap_mode, cudaStream_t st)
{
    k_build_ext<<<dim3((ext_len + 255) / 256, n_sats * 4), 256, 0, st>>>(C, Ep, n_sats, Q, ext_len, wrap_mode);
    return 1;
}

// Grid of a search launch = the number of its CTAs that store cells (clusters: rank 0 stores for its cluster).
// launch_search* and the host's SearchArgs::ctas_total both come from here.
// Which C/A search kernel a search runs: non-coherent sums -> k_search_l1_multi (code run resident in tensor memory);
// K = 1 on full bins -> k_search_l1_cr (capture residue resident in tensor memory, chunks of tiles claimed); K = 1 on
// half-bins -> k_search_l1<false> (odd and even half-bins read different capture spectra: nothing could stay resident).
// k_search_l1_dr (one CTA per SM, two teams with staging warps, capture residue resident, contiguous team ranges) was the
// K = 1 full-bin kernel for most of round 2: +4.7 % over k_search_l1<false> ON THE STATIC STRIDE (6.30 -> 6.02 ms,
// 128-capture farm).  Most of that turned out to be the static stride's own loss -- the two CTAs of an SM run at
// different rates (see claim_tile) -- which the two-team CTA happened not to have: with claimed tiles k_search_l1<false>
// does the same farm in 5.78 ms, k_search_l1_dr in 5.96 ms, and k_search_l1_cr -- the resident capture residue in the
// two-CTA form, residue loop fully unrolled at 126 registers -- in 5.24 ms (32.1 M tiles/s).  On the reference's
// one-capture search: 70.9 us through acq_search against 75.4 us (k_search_l1<false>) and 77.5 us (k_search_l1_dr).
// k_search_l1_dr is compiled only into variant libraries, for the equivalence tests and A/B runs: ACQ_DR_MIN_TILES_PER_SM
// >= 0 (l1_dr_all = 0, l1_dr12 = 12) sends full-bin K = 1 searches of at least that many tiles per SM to it.
#ifndef ACQ_FORCE_L1_CTA
#define ACQ_FORCE_L1_CTA 0   // variant l1_cta: always k_search_l1<false> for K = 1 (the kernel-equivalence tests)
#endif
#ifndef ACQ_DR_MIN_TILES_PER_SM
#define ACQ_DR_MIN_TILES_PER_SM -1   // product: never
#endif
constexpr int kDrMinTilesPerSm = ACQ_DR_MIN_TILES_PER_SM;
#ifndef ACQ_L1_CR
#define ACQ_L1_CR 1   // 0 (variant l1_nocr): full-bin K = 1 searches on k_search_l1<false>
#endif
bool search_claims_tiles(long long n_tiles, int grid);
int search_kind_l1(int K, int half_bin, long long n_tiles, int sm_count)
{
#if defined(ACQ_VARIANT_L1_X3) || defined(ACQ_VARIANT_L1_LDG) || defined(ACQ_VARIANT_L1_MULTI_TW)
    return kSearchL1;   // these experiment builds run every C/A search on their own 256-thread kernels
#endif
#ifdef ACQ_VARIANT_L1_MST
    if (K > 1) return kSearchL1Mst;
#endif
    if (K > 1) return kSearchL1Multi;
    if (half_bin || ACQ_FORCE_L1_CTA) return kSearchL1;
    if (kDrMinTilesPerSm >= 0) return n_tiles < (long long)kDrMinTilesPerSm * sm_count ? kSearchL1 : kSearchL1Dr;
    // full bins: the capture-resident kernel (chunks claimed from six rounds of tiles per CTA up, static stride below)
    return ACQ_L1_CR ? kSearchL1Cr : kSearchL1;
}

// Claimed tiles or the static stride?  Claiming evens out the two CTAs of an SM and the SMs among themselves, at the price
// of a greedy tail: once the counter runs dry every CTA still finishes its tile, up to a whole tile time with the SM half
// empty.  Over many rounds that is noise against what the balance wins (13.7 rounds of E1B tiles: 201.6 -> 190.5 us through
// acq_search; K = 20: 3.65 -> 3.45 ms); the reference's own C/A search is 4.4 rounds, where the static stride's fixed
// pattern (the early CTA of each SM runs five tiles, the late one four, the last of them alone) ends 3.6 us sooner
// (75.4 against 79.0 us, hot caches).  ACQ_DYN_MIN_ROUNDS: rounds (tiles per CTA) from which a launch claims.
#ifndef ACQ_DYN_MIN_ROUNDS
#define ACQ_DYN_MIN_ROUNDS 6
#endif
bool search_claims_tiles(long long n_tiles, int grid)
{
    return grid > 0 && n_tiles >= (long long)ACQ_DYN_MIN_ROUNDS * grid;
}

// Chunk schedule of k_search_l1_cr: runs of 16 tiles, then of 4, then single tiles -- the last two rounds of the launch
// (2 x grid tiles) go out one by one and the two rounds' worth before them in fours, so the tail stays one tile long.
void search_chunks(long long n_tiles, int grid, unsigned *n16, unsigned *n4)
{
    *n16 = *n4 = 0;
    if (!search_claims_tiles(n_tiles, grid)) return;   // static stride: single tiles, tile = blockIdx.x + i gridDim.x
    const long long singles = 2LL * grid, mids = 2LL * kCkMid * grid;
    long long t2 = n_tiles - singles;
    if (t2 < 0) t2 = 0;
    long long t1 = t2 - mids;
    if (t1 < 0) t1 = 0;
    t1 -= t1 % kCkBig;
    *n16 = (unsigned)(t1 / kCkBig);
    *n4 = (unsigned)((t2 - t1) / kCkMid);
}
long long search_chunk_count(long long n_tiles, int grid)
{
    unsigned n16, n4;
    search_chunks(n_tiles, grid, &n16, &n4);
    return (long long)n16 + n4 + (n_tiles - (long long)kCkBig * n16 - (long long)kCkMid * n4);
}

void search_chunk_lengths(int *big, int *mid)
{
    *big = (int)kCkBig;
    *mid = (int)kCkMid;
}

int search_grid_ctas(long long n_tiles, int kind, int sm_count)
{
    if (n_tiles <= 0 || n_tiles > kMaxTilesPerLaunch) return 0;
    if (kind == kSearchL1Cr) {
        const long long chunks = search_chunk_count(n_tiles, 2 * sm_count);
        return (int)(chunks < 2LL * sm_count ? chunks : 2LL * sm_count);
    }
    long long cap = (long long)sm_count * 2;  // two persistent CTAs per SM
    if (kind == kSearchE1bCluster) cap = sm_count / 4;
    if (kind == kSearchL1Dr || kind == kSearchL1Mst) cap = sm_count;   // one CTA per SM, two teams in it
#ifdef ACQ_VARIANT_L1_X3
    if (kind == kSearchL1) cap = (long long)sm_count * 3;
#endif
    return (int)(n_tiles < cap ? n_tiles : cap);
}

// Which searches have an aided form: those that run on the product's search kernels (search_aided_supported).
bool search_aided_supported(int K, int half_bin, long long tiles_l1, long long tiles_e1b, int sm_count)
{
#if defined(ACQ_VARIANT_L1_X3) || defined(ACQ_VARIANT_L1_LDG) || defined(ACQ_VARIANT_L1_MULTI_TW)
    if (tiles_l1 > 0) return false;
#endif
#ifdef ACQ_VARIANT_E1B_LDG
    if (tiles_e1b > 0) return false;
#endif
    (void)tiles_e1b;
    if (tiles_l1 <= 0) return true;
    const int kind = search_kind_l1(K, half_bin, tiles_l1, sm_count);
    return kind == kSearchL1 || kind == kSearchL1Multi || kind == kSearchL1Cr;
}

// The aided instantiations of the product search kernels (launch_search with SearchArgs::dop_center set).
static int launch_search_aided(const AidedSearchArgs &a, int kind, int grid, bool e1b, int sm_count, cudaStream_t st, bool pdl)
{
    using A = AidedSearchArgs;
    if (e1b) {
        if (a.K > 1) launch_k(k_search_e1b_multi<A>, grid, 256, e1b_multi_smem_bytes(), st, pdl, a);
        else launch_k(k_search_e1b<A>, grid, 256, search_e1b_smem_bytes(), st, pdl, a);
    } else if (a.K > 1) {
        launch_k(k_search_l1_multi<A>, grid, 256, l1_multi_smem_bytes(), st, pdl, a);
    } else if (kind == kSearchL1Cr) {
        AidedSearchArgs c = a;
        search_chunks(c.n_tiles, 2 * sm_count, &c.ck_n16, &c.ck_n4);
        launch_k(k_search_l1_cr<A>, grid, 256, l1_multi_smem_bytes(), st, pdl, c);
    } else {
        launch_k(k_search_l1<false, A>, grid, 256, search_l1_smem_bytes(), st, pdl, a);
    }
    return 1;
}

int launch_search(const SearchArgs &a_in, bool e1b, int sm_count, cudaStream_t st, bool pdl)
{
    const int kind = e1b ? kSearchE1b : search_kind_l1(a_in.K, a_in.half_bin, a_in.n_tiles, sm_count);
    const int grid = search_grid_ctas(a_in.n_tiles, kind, sm_count);
    if (grid <= 0) return 0;
    SearchArgs a = a_in;
    if (!search_claims_tiles(a.n_tiles, grid)) a.tile_ctr = nullptr;   // few rounds: static stride
    if (a.dop_center) return launch_search_aided(AidedSearchArgs(a), kind, grid, e1b, sm_count, st, pdl);
    using S = SearchArgs;
    if (e1b) {
#ifdef ACQ_VARIANT_E1B_LDG
        launch_k(k_search_e1b_ldg, grid, 256, fft_smem3_bytes() + 64 * sizeof(float), st, pdl, a);
#else
        if (a.K > 1) launch_k(k_search_e1b_multi<S>, grid, 256, e1b_multi_smem_bytes(), st, pdl, a);
        else launch_k(k_search_e1b<S>, grid, 256, search_e1b_smem_bytes(), st, pdl, a);
#endif
        return 1;
    }
#if defined(ACQ_VARIANT_L1_X3)
    launch_k(a.K > 1 ? k_search_l1_x3<true> : k_search_l1_x3<false>, grid, 256, search_l1_x3_smem(), st, pdl, a);
#elif defined(ACQ_VARIANT_L1_LDG)
    launch_k(a.K > 1 ? k_search_l1_ldg<true> : k_search_l1_ldg<false>, grid, 256, fft_smem3t_bytes() + 64 * sizeof(float), st,
             pdl, a);
#elif defined(ACQ_VARIANT_L1_MULTI_TW)   // the K > 1 form that keeps the stage-B twiddles (not the code run) in tensor memory
    launch_k(a.K > 1 ? k_search_l1<true, S> : k_search_l1<false, S>, grid, 256, search_l1_smem_bytes(), st, pdl, a);
#else
#ifdef ACQ_VARIANT_L1_MST
    if (kind == kSearchL1Mst) launch_k(k_search_l1_mst, grid, kStThreads, dr_smem_bytes(), st, pdl, a);
    else
#endif
    if (a.K > 1) launch_k(k_search_l1_multi<S>, grid, 256, l1_multi_smem_bytes(), st, pdl, a);
    else if (kind == kSearchL1Cr) {
        search_chunks(a.n_tiles, 2 * sm_count, &a.ck_n16, &a.ck_n4);
        launch_k(k_search_l1_cr<S>, grid, 256, l1_multi_smem_bytes(), st, pdl, a);
    }
#if defined(ACQ_VARIANT_L1_SP)
    else if (kind == kSearchL1Dr) launch_k(k_search_l1_sp, grid, kSpThreads, sp_smem_bytes(), st, pdl, a);
#elif defined(ACQ_VARIANT_L1_ST)
    else if (kind == kSearchL1Dr) launch_k(k_search_l1_st, grid, kStThreads, st_smem_bytes(), st, pdl, a);
#endif
#if ACQ_DR_MIN_TILES_PER_SM >= 0
    else if (kind == kSearchL1Dr) launch_k(k_search_l1_dr, grid, kStThreads, dr_smem_bytes(), st, pdl, a);
#endif
    else launch_k(k_search_l1<false, S>, grid, 256, search_l1_smem_bytes(), st, pdl, a);
#endif
    return 1;
}

int launch_search_e1b_cluster(const SearchArgs &a, int sm_count, cudaStream_t st, bool pdl)
{
    const int n_clusters = search_grid_ctas(a.n_tiles, kSearchE1bCluster, sm_count);
    if (n_clusters <= 0) return 0;
    if (a.dop_center)
        launch_k(a.K > 1 ? k_search_e1b_cluster<true, AidedSearchArgs> : k_search_e1b_cluster<false, AidedSearchArgs>, 4 * n_clusters,
                 256, search_e1b_cluster_smem_bytes(), st, pdl, AidedSearchArgs(a));
    else
        launch_k(a.K > 1 ? k_search_e1b_cluster<true, SearchArgs> : k_search_e1b_cluster<false, SearchArgs>, 4 * n_clusters, 256,
                 search_e1b_cluster_smem_bytes(), st, pdl, a);
    return 1;
}

int launch_refine(const float2 *Dp, const float2 *Ep, const acq_record *rec, const int *sat_type, acq_fine *out, int n_rows,
                  int n_slots, int K, int nvar, int half_bin, int ext_len, int Q, int n_shift, int smax, int cd_div,
                  cudaStream_t st)
{
    if (n_rows <= 0) return 0;
    RefineArgs a{Dp, Ep, rec, sat_type, out, n_slots, K, nvar, half_bin, ext_len, Q, n_shift, smax, cd_div};
    k_refine<<<n_rows, 256, 0, st>>>(a);
    return 1;
}

#ifdef ACQ_TRACE
}  // namespace acq
// variant "trace" only: copies the stamps out ([kernel][cta][slot], ns of %globaltimer) and clears them
extern "C" int acq_trace_read(unsigned long long *out, int n)
{
    const int total = acq::kTraceKernels * acq::kTraceCtas * 4;
    if (!out || n < total) return total;
    if (cudaMemcpyFromSymbol(out, acq::g_trace, sizeof(unsigned long long) * total) != cudaSuccess) return -1;
    static unsigned long long zero[acq::kTraceKernels * acq::kTraceCtas * 4];
    cudaMemcpyToSymbol(acq::g_trace, zero, sizeof zero);
    return total;
}
namespace acq {
#endif

int launch_best_dop(const acq_cell *cells, const int *slot_sat, acq_record *out, int n_cap, int n_slots, int n_dop,
                    PickDop pd, cudaStream_t st, bool pdl)
{
    const int n_rows = n_cap * n_slots;
    launch_k(k_best_dop, (n_rows + 3) / 4, 128, 0, st, pdl, cells, slot_sat, out, n_rows, n_slots, n_dop, pd);
    return 1;
}

int launch_pick_small(const acq_cell *cells, const int *slot_sat, acq_record *out, unsigned *ctas_done, unsigned ctas_total,
                      unsigned *host_flag, unsigned epoch, int n_rows, int n_slots, int n_dop, PickDop pd, cudaStream_t st,
                      bool pdl)
{
    launch_k(k_pick_small, 1, 1024, 0, st, pdl, cells, slot_sat, out, ctas_done, ctas_total, host_flag, epoch, n_rows, n_slots,
             n_dop, pd);
    return 1;
}

}  // namespace acq
