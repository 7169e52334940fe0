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
#include <type_traits>

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
    pdl_launch_dependents();
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
    pdl_launch_dependents();
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
    // Doppler index h of the tile: dop_lo + d, or in an aided search (AidedSearchArgs) d steps into its row's window.  The
    // claiming kernels form a tile's indices in the one thread that publishes them, so the centre's load stays there.
    template <class PA>
    __device__ __forceinline__ void set_dop(const PA &p)
    {
        int h;
        if constexpr (PA::kCoh) {   // 1/F-bin steps: integer bin (floored) and sub-bin variant
            // an aided coherent search (AidedCohSearchArgs): the window and dop_lo..dop_hi in the same 1/F-bin units
            if constexpr (PA::kAided) h = window_lo(__ldg(p.dop_center + cap * p.n_slots + slot), p.half_width, p.dop_lo, p.dop_hi) + d;
            else h = p.dop_lo + d;
            const int F = p.nvar;
            dop = (h >= 0 ? h : h - F + 1) / F;
            v = h - F * dop;
            return;
        }
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
    // (an aided coherent search: F = nvar steps per bin; unreached, acq_api.cu refuses coherent code_doppler searches)
    int h;
    if constexpr (PA::kAided && PA::kCoh) h = ti.dop * p.nvar + ti.v;
    else if constexpr (PA::kAided) h = ti.dop * (1 + p.half_bin) + ti.v;
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
// B->C tiles live inside the exchange rows.  The L2 round trip is off every warp's dependent chain (a form that loaded
// both operands straight from L2 was measured 7 % slower on cfg2); 98.6 KiB of shared memory per CTA, two CTAs per SM.
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
    pdl_launch_dependents();
    // thread 0: stage the operands of sub-FFT (tn, bn, k2n) -- D into S1 half `half`, E into the E buffer
    auto issue = [&](const TileIdx &tn, int bn, int k2n, int half) {
        const int r = (k2n - tn.dop) & 3;
        const int q = (k2n - tn.dop - r) >> 2;
        const float2 *Dk = p.Dp + d_row(p, tn, bn) * kN + k2n * kSub;
        const float2 *Ek = p.Ep + (size_t)(tn.sat * 4 + r) * p.ext_len + ((p.Q + q) & ~1);
        fence_proxy_async();  // generic-proxy reads of these buffers (ordered by the CTA barrier) before the async writes
        mbar_expect_tx(bar, (uint32_t)(sizeof(float2) * (kSub + kEBufElems)));
        tma_load_1d(smem_u32(s.E), Ek, (uint32_t)(sizeof(float2) * kEBufElems), bar);
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
                    const float2 *Ek = s.E + ((p.Q + q) & 1) + t;
                    mbar_wait(bar, (uint32_t)(it & 1));
#pragma unroll
                    for (int a = 0; a < 16; a++) x[a] = cmul_conj_a(Dk[kRowElems * a], Ek[256 * a]);
                }
                subfft4096_inv4(x, k2, bw, S1b, t, tw_taddr, [&]() {
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
        warp_reduce_peak_redux(thread_peak_l1(P, t), red_f + 16 * par, red_i + 8 * par, t);
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
    pdl_launch_dependents();
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

// k_search_l1_coh -- coherent search (acq_search_coherent): k_search_l1_multi's tile (code run E resident in tensor memory
// across the K blocks, D staged per block by TMA, same sub-FFTs and combine), but the K blocks form G = K / M groups of M
// and the lag vectors of a group are added as complex numbers before any power is taken.
//   Block j of a group is rotated by exp(i theta_j), theta_j = 2 pi j (v / F - 16 d / N): the carrier phase that block's
//   processing removed.  A carrier exp(2 pi i (d + v / F) n / N) (the signal Doppler index h = F d + v selects; see the
//   front end's conventions) advances by d + v / F cycles per 16384-sample block; the sub-bin rotation restarts every block
//   and so leaves v / F cycles per block, the integer d cycles vanish, and the 16 b-sample circular delay that lines the
//   code up (k_front_end) moves the block's carrier back by 16 b d / N cycles.  The correlation conj(D) C carries the
//   conjugate phase, so r'_b ~ exp(-2 pi i b (v / F - 16 d / N)) and theta_j undoes it.  theta_0 = 0: block 0 of a group
//   is used as computed.
//   Data-bit hypotheses: T = sum of the group's rotated blocks u_j, prefixes S_s = sum_{j<s} u_j (s = 1..M-1); a bit
//   edge before block s gives |S_s - (T - S_s)|^2 = |2 S_s - T|^2, no edge |T|^2; the group adds max over the M
//   hypotheses into P.  The prefixes live in tensor memory: the thread's 128 columns next to the code run (512 columns
//   per CTA, so one CTA per SM; 255 registers for T, P, the accumulators and the sub-FFT operands).
//   M = 1: one hypothesis, P[n] = sum_b |r'_b[n]|^2 with k_search_l1_multi's operations in its order: the same cells.
#ifndef ACQ_COH_UNROLL
#define ACQ_COH_UNROLL 4
#endif
template <class PA>
__global__ void __launch_bounds__(256, 1) k_search_l1_coh(const PA p)
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
    constexpr int L = ACQ_LAGS_L1;
    const int M = p.m_coh;
    const int FN = p.nvar * kN;   // phase unit: 1 / (F N) cycle
    const uint32_t tmem_base = tmem_alloc_cta<4 * kTwCols>(reinterpret_cast<uint32_t *>(red_f + 48), t);
    const uint32_t e_taddr = tmem_base + tmem_lane_base(t) + (uint32_t)((t >> 7) * 2 * kTwCols);  // [k2][16 complex]
    const uint32_t s_taddr = e_taddr + kTwCols;                                                   // [s - 1][16 complex]
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
    pdl_launch_dependents();
    auto issue = [&](const TileIdx &tn, int bn, int k2n, int half) {
        const int r = (k2n - tn.dop) & 3;
        const int q = (k2n - tn.dop - r) >> 2;
        const float2 *Dk = p.Dp + d_row(p, tn, bn) * kN + k2n * kSub;
        fence_proxy_async();
        if (bn == 0) {
            const float2 *Ek = p.Ep + (size_t)(tn.sat * 4 + r) * p.ext_len + ((p.Q + q) & ~1);
            mbar_expect_tx(bar, (uint32_t)(sizeof(float2) * (kSub + kEBufElems)));
            tma_load_1d(smem_u32(s.E), Ek, (uint32_t)(sizeof(float2) * kEBufElems), bar);
        } else {
            mbar_expect_tx(bar, (uint32_t)(sizeof(float2) * kSub));
        }
        tma_load_1d(smem_u32(s.S1 + half * kSub), Dk, (uint32_t)(sizeof(float2) * kSub), bar);
    };
    TileIdx ti(p, blockIdx.x);
    if (t == 0) issue(ti, 0, 0, 0);
    int *feed = red_i + 20;
    unsigned nxt = blockIdx.x;
    int it = 0;
    int par = 0, pend_cap = -1, pend_slot = 0, pend_d = 0;
    auto flush = [&]() {
        store_cell(p, pend_cap, pend_slot, pend_d, merge_warp_peaks(red_f + 16 * (par ^ 1), red_i + 8 * (par ^ 1)), L);
    };

    for (;;) {
        float P[16];
        float2 acc[16], T[16];
        // theta_j of this tile in units of 1 / (F N) cycle: j * (v N - 16 d F) mod F N
        int step = (ti.v * kN - 16 * ti.dop * p.nvar) % FN;
        if (step < 0) step += FN;
        int j = 0, ph = 0;
        for (int b = 0; b < p.K; b++) {
            float2 x[16];
            constexpr int kCohUnroll = ACQ_COH_UNROLL;
#pragma unroll kCohUnroll
            for (int k2 = 0; k2 < 4; k2++) {
                float2 *S1b = s.S1 + (it & 1) * kSub;
                const float2 *Dk = S1b + t;
                if (b == 0) {
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
#pragma unroll
                for (int a = 0; a < 16; a++) x[a] = cmul_conj_a(Dk[256 * a], x[a]);
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
                if (t == 0 && b == 0 && k2 == 0 && pend_cap >= 0) flush();
                if (k2 == 0) {
#pragma unroll
                    for (int n2 = 0; n2 < 16; n2++) acc[n2] = x[r16(n2)];
                } else {
#pragma unroll
                    for (int n2 = 0; n2 < 16; n2++) acc[n2] = cfma(x[r16(n2)], c_cC[k2][n2], acc[n2]);
                }
            }
            if (j == 0) {
#pragma unroll
                for (int n2 = 0; n2 < 16; n2++) T[n2] = acc[n2];
            } else {   // S_j = T, then T += exp(i theta_j) r'_b
                tmem_st16(s_taddr + 32 * (j - 1), T);
                tmem_wait_st();
                float sn, cs;
                sincospif(__fdiv_rn((float)(2 * ph), (float)FN), &sn, &cs);
                const float2 w = make_float2(cs, sn);
#pragma unroll
                for (int n2 = 0; n2 < 16; n2++) T[n2] = cfma(acc[n2], w, T[n2]);
            }
            if (j == M - 1) {   // end of the group: best data-bit hypothesis per lag
                float pg[16];
#pragma unroll
                for (int n2 = 0; n2 < 16; n2++) pg[n2] = cpower(T[n2]);
                for (int e = 1; e < M; e++) {
                    float2 S[16];
                    tmem_ld16(s_taddr + 32 * (e - 1), S);
                    tmem_wait_ld();
#pragma unroll
                    for (int n2 = 0; n2 < 16; n2++)
                        pg[n2] = fmaxf(pg[n2], cpower(make_float2(2.0f * S[n2].x - T[n2].x, 2.0f * S[n2].y - T[n2].y)));
                }
#pragma unroll
                for (int n2 = 0; n2 < 16; n2++) P[n2] = (b == M - 1) ? pg[n2] : (P[n2] + pg[n2]);
                j = 0;
                ph = 0;
            } else {
                j++;
                ph += step;
                if (ph >= FN) ph -= FN;
            }
        }
        warp_reduce_peak(thread_peak_l1(P, t), red_f + 16 * par, red_i + 8 * par, t);
        pend_cap = ti.cap;
        pend_slot = ti.slot;
        pend_d = ti.d;
        par ^= 1;
        if (!next_tile(feed, ti)) break;
    }
    __syncthreads();
    if (t == 0 && pend_cap >= 0) flush();
    claims_done(p, t);
    search_cta_epilogue(p, t);
    tmem_free_cta<4 * kTwCols>(tmem_base, t);
}

// Sub-bin variants of a coherent search: variant v (1..F-1) of block row r = variant 0 (k_front_end's output, delayed by
// 16 (r mod K) samples) times rot[v][o] at the sample's undelayed index o, with the half-bin variant's arithmetic, so
// variant F/2 of an even F is bit-identical to the half-bin variant of k_front_end.
__global__ void __launch_bounds__(256) k_coh_variants(float2 *__restrict__ x2, const float2 *__restrict__ rot, int F, int K,
                                                      int row0)
{
    const int m = blockIdx.x * 256 + threadIdx.x;
    float2 *row = x2 + (size_t)blockIdx.y * F * kN;
    const int o = (m - 16 * ((row0 + (int)blockIdx.y) % K)) & (kN - 1);
    const float2 y = row[m];
    for (int v = 1; v < F; v++) {
        const float2 w = __ldg(rot + (size_t)v * kN + o);
        row[(size_t)v * kN + m] = make_float2(__fsub_rn(__fmul_rn(y.x, w.x), __fmul_rn(y.y, w.y)),
                                              __fadd_rn(__fmul_rn(y.x, w.y), __fmul_rn(y.y, w.x)));
    }
}

// k_search_l1_cr -- K = 1 on full bins with the CAPTURE operand resident in tensor memory and tiles claimed in CHUNKS.
// A thread always reads the same 16 values of a capture residue: 4 residues x 16 complex = its 128 TMEM columns, so D is
// staged and parked once per capture and comes back by one tcgen05.ld per sub-FFT.  Two CTAs per SM; a CTA draws runs
// of consecutive tiles (same capture, bar the boundaries), 16 tiles long while the launch is young, 4 and then single
// tiles towards its end (SearchArgs::ck_n16 / ck_n4, search_chunks()), so the greedy tail stays one tile long while D is
// re-staged for ~1 tile in 14.  Stage-B twiddles: the 7.5 KiB shared table;
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
// four (28.1 / 30.6 / 32.1 M tiles/s; k_search_l1<false> with claimed tiles: 5.78 ms, the two-team staging-warp kernel of
// round 2: 5.96 ms).
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
    pdl_launch_dependents();
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
    pdl_launch_dependents();
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
        // radix-4 combine over k2, lags n = lag_of3(t, n2) + 4096 m < 16368.  A thread's lags grow with n2 inside a
        // quarter m and with m across quarters: one running (max, n2) per quarter with a strict >, merged in the order
        // m = 0..3 with a strict >, keeps the first maximum (search.cpp:488) without comparing indices.
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
    pdl_launch_dependents();
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
// grain than k_search_e1b.  The host picks the form in acq_api.cu (variants e1b_cta / e1b_cluster force one).
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
    pdl_launch_dependents();

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

#ifdef ACQ_VARIANT_E1B_LDG
// k_search_e1b_ldg: the one-CTA E1B search with operands read straight from L2 and a reduction barrier per tile -- the
// reference k_search_e1b is tested against (variant library e1b_ldg; the product library does not contain it).
__global__ void __launch_bounds__(256, 2) k_search_e1b_ldg(const SearchArgs p)
{
    extern __shared__ __align__(1024) unsigned char smem[];
    const FftSmem3 s = fft_smem3_carve(smem);
    float *red_f = reinterpret_cast<float *>(smem + fft_smem3_bytes());
    int *red_i = reinterpret_cast<int *>(red_f + 16);
    const int t = threadIdx.x;
    constexpr int L = ACQ_LAGS_E1B;
    const uint32_t tmem_base = tmem_alloc_cta<kE1bTmemCols>(reinterpret_cast<uint32_t *>(red_f + 32), t);
    load_t2(s, p.tables, t);
    // this thread's scratch: lane 32*(warp%4) + (t%32), columns [96*(warp/4), +96): [k2][n2] complex
    const uint32_t zaddr = tmem_base + tmem_lane_base(t) + (uint32_t)((t >> 7) * 96);
    const float2 *base = p.tables + kT2Elems + t;
    int buf = 0;
    if (p.wait_prior) pdl_wait();
    pdl_launch_dependents();  // after the wait (see k_search_l1)

    for (long long tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x) {
        const TileIdx ti(p, tile);
        float2 x[16];
#pragma unroll 1
        for (int k2 = 0; k2 < 4; k2++) {
            load_products(x, p, ti, 0, k2, t);
            subfft4096_inv3(x, k2, __ldg(base + k2 * 256), buf, s, t);
            buf ^= 1;
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
        const Peak tot = block_reduce_peak(best, red_f, red_i, t);
        if (t == 0) store_cell(p, ti.cap, ti.slot, ti.d, tot, L);
    }
    __syncthreads();
    search_cta_epilogue(p, t);
    tmem_free_cta<kE1bTmemCols>(tmem_base, t);
}

#endif  // ACQ_VARIANT_E1B_LDG

// ---------------------------------------------------------------------------------------------
// K6.  Hand-off to tracking: refinement (k_refine: acq_refine*, acq_refine_coherent*) and peak quality (k_profile:
// acq_profile*, acq_profile_coherent*) of the records of the most recent search, one 256-thread CTA per record, straight
// from the spectra the search left in HBM.  Each kernel has an instance for the records of a non-coherent search
// (RefineArgs / ProfileArgs) and one for those of a coherent search (RefineCohArgs / ProfileCohArgs, kCoh).  The
// non-coherent instance is the coherent arithmetic with M the constant 1, so it compiles none of the group code.
//   A record's dop is an index h of the 1/F-bin grid, F = nvar spectrum variants per block (1 + half_bin; coherent: M (1 +
// half_bin)): code row d = floor(h / F), variant v = h - F d.  Block b of that Doppler index is spectrum row ((cap K + b)
// nvar + v) n_shift + smax + cshift (d_row's rule; cshift: the code-Doppler copy, non-coherent only), which the front end
// delayed by 16 b + cshift samples so that lag n lines up across blocks.  Coherent groups hold blocks b = g M + j; block
// j >= 1 enters its group's sum rotated by theta_j = 2 pi j (v N - 16 d F) / (F N), the phase k_search_l1_coh uses.
//   The records may come from device memory the host never saw (the _device forms), so each CTA first checks its own
// record (record_marker) and a CTA whose record fails a check, or that the DETECTED flag skips, writes a marker row and
// exits before any load of the spectra (a uniform branch: every thread reads the same record).  A coherent record is
// checked on the range M dop_lo .. M dop_hi, and the caller's min_snr arrives as thr_l1 with the DETECTED flag.
// ---------------------------------------------------------------------------------------------
// The checks of the host forms (check_records), in their order, on a record the host may never have seen: 0 if the record
// passes, -2 if it fails one (the satellite's range is checked before sat_type is indexed with it), -1 if `detected_only`
// and it is below its type's threshold.
__device__ __forceinline__ int record_marker(const acq_record &rc, const int *slot_sat, int slot, const int *sat_type, int n_sats,
                                             int dop_lo, int dop_hi, bool detected_only, float thr_l1, float thr_e1b)
{
    int marker = 0;
    if (rc.sat < 0 || rc.sat >= n_sats || rc.sat != slot_sat[slot]) {
        marker = -2;
    } else {
        const bool e1b = sat_type[rc.sat] == ACQ_E1B;
        const int L = e1b ? ACQ_LAGS_E1B : ACQ_LAGS_L1;
        if (rc.lag < 0 || rc.lag >= L) marker = -2;
        // a row that never exceeded snr 0 carries dop 0 (k_best_dop), which may lie outside an asymmetric range
        else if ((rc.dop < dop_lo || rc.dop > dop_hi) && !(rc.dop == 0 && rc.snr == 0.0f)) marker = -2;
        else if (detected_only && !(rc.snr >= (e1b ? thr_e1b : thr_l1))) marker = -1;
    }
    return marker;
}

// Code row d = floor(h / F) of Doppler index h.  F = 1 + half_bin of a non-coherent search floors by a shift: a division
// there moved k_refine's loads behind its twiddle arithmetic (+28 % time) and cost k_profile<E1B> a spill.
template <class A>
__device__ __forceinline__ int code_row(const A &p, int h)
{
    if constexpr (A::kCoh) return (h >= 0 ? h : h - p.nvar + 1) / p.nvar;
    else return h >> p.half_bin;
}

// Block b's spectrum at variant v and code-Doppler copy cshift: row ((cap K + b) nvar + v) n_shift + smax + cshift (d_row's
// rule).  A coherent search has one copy per spectrum (code_doppler engines are refused), so n_shift = 1 folds in there.
template <class A>
__device__ __forceinline__ const float2 *spectrum_row(const A &p, int cap, int b, int v, int cshift)
{
    const int n_shift = A::kCoh ? 1 : p.n_shift, smax = A::kCoh ? 0 : p.smax;
    return p.Dp + (((size_t)((size_t)cap * p.K + b) * p.nvar + v) * n_shift + (smax + cshift)) * kN;
}

// k_refine (SURVEY 8(f) rank 4).  The search reports the code phase in /DECIM samples and the Doppler in bins of 249.76 Hz
// (search.cpp:574-575); the tracking loops then need a 5 s settle to pull in the LO (gps/channel.cpp:345-372) because
// +-125 Hz exceeds the Costas pull-in range.  For each record this kernel evaluates the correlation
// r_h[n] = sum_k conj(D[k]) C[k-d] e^{+j 2 pi k n / N} (the very sum the inverse FFT computes, search.cpp:471-481) at five
// points around the peak -- (h - H, n) (h, n - 1) (h, n) (h, n + 1) (h + H, n), H = F / M: one bin of the group's DFT
// (ACQ_BIN_HZ / M) -- each Doppler point at its own (d', v') = split(h +- H), so at M > 1 it reads its own spectrum
// variant and code row (at M = 1 the three points share v and d' = d -+ 1).  Thread 0 folds block j of a group into each
// point's group sum rotated by that point's theta_j, keeps the prefixes, and at the group's end applies the data-bit
// hypothesis that is the first maximum at the centre point (h, n) -- "no edge", then s = 1..M-1, the search's rule -- to
// all five sums.  A code row shifted by d' puts e^{+j 2 pi d' n_b / N} on a block's sum at lag n_b = n + 16 b + cshift;
// theta_j removes the 16 j d' part, so a group sum carries that of its first block, n_b0 = n + 16 (b - j) + cshift, and
// the outer points are put back on the centre's phase by e^{-+j 2 pi (d' - d) n_b0 / N} where d' != d (the spectrum
// variants rotate at the undelayed sample index, k_coh_variants, and add no lag-dependent phase).  Then, summed over the
// groups:
//   Doppler: delta = Re[(Xm - Xp) conj(2 X0 - Xm - Xp)] / |2 X0 - Xm - Xp|^2   (three-bin interpolation of a
//            rectangular-window DFT), dop_hz = (h / F + delta / M) ACQ_BIN_HZ,
//   code   : eps = slope (l - e) / (l + e),  e/l = Re(X[n-+1] conj(X[n]))       (early-minus-late over the
//            correlation triangle: 4 samples per chip -> slope 3; BOC(1,1) main peak -> slope 1/3),
//   peak   : sum of |X(h, n)|^2.
// Thread t owns k1 = t + 256 i for all four residues.
template <class RA>
__global__ void __launch_bounds__(256) k_refine(const RA p)
{
    __shared__ float red[8][10];
    __shared__ float2 pre[5][ACQ_COH_MAX - 1];   // coherent, thread 0: prefixes S_s of the five group sums
    const int row = blockIdx.x, t = threadIdx.x;
    const acq_record rc = p.rec[row];
    const int cap = row / p.n_slots;
    const int marker = record_marker(rc, p.slot_sat, row % p.n_slots, p.sat_type, p.n_sats, p.dop_lo, p.dop_hi,
                                     (p.flags & ACQ_REFINE_DETECTED) != 0, p.thr_l1, p.thr_e1b);
    if (marker != 0) {
        if (t == 0) {
            acq_fine o;
            o.dop_hz = o.code_fs = __int_as_float(0x7fc00000);   // quiet NaN
            o.peak = 0.0f;
            o.ca_shift = marker;
            p.out[row] = o;
        }
        return;
    }
    // every row of a coherent search is C/A (reading its type moved the coherent instance's loads: +5 % time)
    const bool e1b = !RA::kCoh && p.sat_type[rc.sat] == ACQ_E1B;
    int M = 1;
    if constexpr (RA::kCoh) M = p.m_coh;
    const int F = p.nvar, H = F / M, FN = F * kN;
    const int n = rc.lag;
    int dd[3], vv[3], step[3], ph[3];   // Doppler points h - H, h, h + H: code row, variant, theta step, phase
#pragma unroll
    for (int i = 0; i < 3; i++) {
        const int hh = rc.dop + (i - 1) * H;
        dd[i] = code_row(p, hh);
        vv[i] = hh - F * dd[i];
        step[i] = (vv[i] * kN - 16 * dd[i] * F) % FN;
        if (step[i] < 0) step[i] += FN;
        ph[i] = 0;
    }
    float num = 0.0f, den = 0.0f, early = 0.0f, late = 0.0f, peak = 0.0f;  // thread 0 only
    float2 T[5];                                                           // thread 0 only: the group sums
    for (int b = 0; b < p.K; b++) {
        const int j = b % M;
        const int cshift = !RA::kCoh && p.n_shift > 1 ? code_shift(b, rc.dop, p.cd_div) : 0;
        const float2 *D0 = spectrum_row(p, cap, b, vv[1], cshift);
        const float2 *Dm = RA::kCoh ? spectrum_row(p, cap, b, vv[0], 0) : D0;
        const float2 *Dp = RA::kCoh ? spectrum_row(p, cap, b, vv[2], 0) : D0;
        float2 acc[5];
#pragma unroll
        for (int i = 0; i < 5; i++) acc[i] = make_float2(0.0f, 0.0f);
        for (int k2 = 0; k2 < 4; k2++) {
            const float2 *Er[3];
#pragma unroll
            for (int i = 0; i < 3; i++) {  // code rows of the three Doppler points
                const int r = (k2 - dd[i]) & 3;
                const int q = (k2 - dd[i] - r) >> 2;
                Er[i] = p.Ep + (size_t)(rc.sat * 4 + r) * p.ext_len + p.Q + q;
            }
            for (int k1 = t; k1 < kSub; k1 += 256) {
                const int k = 4 * k1 + k2;
                float sn, cs, s1, c1;
                sincospif((float)((k * n) & (kN - 1)) * (1.0f / 8192.0f), &sn, &cs);  // e^{+j 2 pi k n / N}
                sincospif((float)k * (1.0f / 8192.0f), &s1, &c1);                      // e^{+j 2 pi k / N}
                const float2 w0 = make_float2(cs, sn), wk = make_float2(c1, s1);
                const float2 pm = cmul(cmul_conj_a(Dm[k2 * kSub + k1], Er[0][k1]), w0);
                const float2 pc = cmul(cmul_conj_a(D0[k2 * kSub + k1], Er[1][k1]), w0);
                const float2 pp = cmul(cmul_conj_a(Dp[k2 * kSub + k1], Er[2][k1]), w0);
                acc[0] = cadd(acc[0], pm);
                acc[1] = cadd(acc[1], cmul(pc, make_float2(c1, -s1)));  // lag n-1
                acc[2] = cadd(acc[2], pc);
                acc[3] = cadd(acc[3], cmul(pc, wk));                    // lag n+1
                acc[4] = cadd(acc[4], pp);
            }
        }
        // CTA reduction of the five complex sums
#pragma unroll
        for (int i = 0; i < 5; i++) {
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) {
                acc[i].x += __shfl_xor_sync(0xffffffffu, acc[i].x, off);
                acc[i].y += __shfl_xor_sync(0xffffffffu, acc[i].y, off);
            }
        }
        __syncthreads();  // red[] of the previous block has been consumed
        if ((t & 31) == 0) {
#pragma unroll
            for (int i = 0; i < 5; i++) {
                red[t >> 5][2 * i] = acc[i].x;
                red[t >> 5][2 * i + 1] = acc[i].y;
            }
        }
        __syncthreads();
        if (t == 0) {
            float2 R[5];
#pragma unroll
            for (int i = 0; i < 5; i++) {
                R[i] = make_float2(0.0f, 0.0f);
                for (int w = 0; w < 8; w++) R[i].x += red[w][2 * i], R[i].y += red[w][2 * i + 1];
            }
            if (j == 0) {
#pragma unroll
                for (int i = 0; i < 5; i++) T[i] = R[i];
            } else {   // S_j = T, then T += exp(i theta_j) R, theta_j of each point's own (d', v')
                float2 w[3];
#pragma unroll
                for (int i = 0; i < 3; i++) {
                    float sn, cs;
                    sincospif(__fdiv_rn((float)(2 * ph[i]), (float)FN), &sn, &cs);
                    w[i] = make_float2(cs, sn);
                }
#pragma unroll
                for (int i = 0; i < 5; i++) {
                    pre[i][j - 1] = T[i];
                    T[i] = cfma(R[i], w[i == 0 ? 0 : (i == 4 ? 2 : 1)], T[i]);
                }
            }
            if (j == M - 1) {
                // the data-bit hypothesis of the centre point: first maximum of |T|^2, |2 S_s - T|^2 (s = 1..M-1)
                float pb = cpower(T[2]);
                int sb = 0;
                for (int e = 1; e < M; e++) {
                    const float2 S = pre[2][e - 1];
                    const float pw = cpower(make_float2(2.0f * S.x - T[2].x, 2.0f * S.y - T[2].y));
                    if (pw > pb) pb = pw, sb = e;
                }
                float2 X[5];
#pragma unroll
                for (int i = 0; i < 5; i++) {
                    X[i] = T[i];
                    if (sb) {   // blocks before the edge +1, from it on -1: 2 S_s - T
                        const float2 S = pre[i][sb - 1];
                        X[i] = make_float2(2.0f * S.x - T[i].x, 2.0f * S.y - T[i].y);
                    }
                }
                float sn, cs;
                sincospif((float)((n + 16 * (b - j) + cshift) & (kN - 1)) * (1.0f / 8192.0f), &sn, &cs);
                const float2 Xm = !RA::kCoh || dd[0] != dd[1] ? cmul(X[0], make_float2(cs, sn)) : X[0];
                const float2 Xp = !RA::kCoh || dd[2] != dd[1] ? cmul(X[4], make_float2(cs, -sn)) : X[4];
                const float2 X0 = X[2];
                const float2 a = csub(Xm, Xp);
                const float2 g = csub(csub(cadd(X0, X0), Xm), Xp);
                num += a.x * g.x + a.y * g.y;
                den += g.x * g.x + g.y * g.y;
                early += X[1].x * X[2].x + X[1].y * X[2].y;
                late += X[3].x * X[2].x + X[3].y * X[2].y;
                peak += X[2].x * X[2].x + X[2].y * X[2].y;
#pragma unroll
                for (int i = 0; i < 3; i++) ph[i] = 0;
            } else {
#pragma unroll
                for (int i = 0; i < 3; i++) {
                    ph[i] += step[i];
                    if (ph[i] >= FN) ph[i] -= FN;
                }
            }
        }
    }
    if (t == 0) {
        float delta = den > 0.0f ? num / den : 0.0f;
        delta = fminf(1.0f, fmaxf(-1.0f, delta));
        float eps = (early + late) > 0.0f ? (e1b ? (1.0f / 3.0f) : 3.0f) * (late - early) / (early + late) : 0.0f;
        eps = fminf(1.0f, fmaxf(-1.0f, eps));
        const int L = e1b ? ACQ_LAGS_E1B : ACQ_LAGS_L1;
        // h / F + delta / M; at F = 1 + half_bin and M = 1 the same value without two divisions on every CTA's tail
        const float h_bins = RA::kCoh ? __fdiv_rn((float)rc.dop, (float)F) : (p.half_bin ? 0.5f : 1.0f) * (float)rc.dop;
        acq_fine o;
        o.dop_hz = (h_bins + (RA::kCoh ? __fdiv_rn(delta, (float)M) : delta)) * (float)ACQ_BIN_HZ;
        o.code_fs = (float)ACQ_DECIM * ((float)n + eps);
        o.peak = peak;
        int cs = (int)lrintf(o.code_fs) % (L * ACQ_DECIM);
        if (cs < 0) cs += L * ACQ_DECIM;
        o.ca_shift = cs;
        p.out[row] = o;
    }
}

// k_profile.  Each record's row is evaluated once more at the record's Doppler index, exactly as the search evaluated it:
// the product of the capture spectrum the search read (variant v, the code-Doppler copy) with the extended code row d
// (the same wrap), four sub-FFTs of 4096 points per block, the search's radix-4 combine -- the running accumulation of
// the C/A kernels, the parked-residue butterfly of the E1B kernels -- and the block powers summed in block order, or for a
// coherent search k_search_l1_coh's group step (coh_fold).  Every step is the search kernels' own arithmetic in their
// order (subfft4096_inv3 computes what subfft4096_inv4 / inv4s compute), so the power at every lag is bitwise the one
// the search reduced: the profile at the record's lag is acq_record.peak and the first maximum of the profile is the
// record's lag.  Then one pass over the lags forms the largest power outside the main lobe (circular distance > excl,
// the lowest lag on ties), the mean power there, and the profile row.
// E1B parks three residues in tensor memory as k_search_e1b does and, for K > 1, keeps the 64 running block sums of a
// thread in a thread-private 64 KiB shared-memory array (the C/A sums stay in registers); the coherent instance keeps the
// group prefixes in tensor memory as the search does (256 columns per CTA: threads t and t + 128 share lanes).  C/A and
// E1B rows of a non-coherent search are two instances launched over the same rows: a CTA whose slot is of the other type
// exits at once.  Every row of a coherent search is C/A.
constexpr size_t kProfileRedBytes = 64 * sizeof(float);                 // reduction slots, the record's power, TMEM slot
constexpr size_t kProfilePsBytes = sizeof(float) * 64 * 256;            // E1B, K > 1: running block sums [64][256]
__host__ __device__ constexpr size_t profile_smem_bytes(bool e1b, int K)
{
    return fft_smem3_bytes() + kProfileRedBytes + (e1b && K > 1 ? kProfilePsBytes : 0);
}
constexpr int kCohPrefixCols = 4 * 32;   // TMEM columns of one thread's prefixes S_1..S_{M-1} (16 complex each)

// One lag of the final powers: the record's power, the running maximum / sum outside the main lobe, the profile.
__device__ __forceinline__ void profile_visit(int n, float pw, int lag, int excl, int L, Peak &best, float *pk, float *prof)
{
    if (n == lag) *pk = pw;
    int d = n - lag;
    d = d < 0 ? -d : d;
    d = min(d, L - d);
    if (d > excl) peak_merge(best, pw, n, pw);   // strict > or the lower lag on equal power
    if (prof) prof[n] = pw;
}

// k_search_l1_coh's group step, in its operations and order: block b, the j-th of its group, with this thread's 16 lag
// values acc.  S_j = T is parked in tensor memory at s_taddr + 32 (j - 1) before T += exp(i theta_j) acc, theta_j =
// 2 pi ph / (F N); at the group's end the best data-bit hypothesis of each lag goes into P, and j / ph advance by one
// block (ph by the record's theta step).  At M = 1 it is P = b == 0 ? |acc|^2 : P + |acc|^2.
__device__ __forceinline__ void coh_fold(const float2 (&acc)[16], float2 (&T)[16], float (&P)[16], int &j, int &ph, int b,
                                         int M, int step, int FN, uint32_t s_taddr)
{
    if (j == 0) {
#pragma unroll
        for (int n2 = 0; n2 < 16; n2++) T[n2] = acc[n2];
    } else {   // S_j = T, then T += exp(i theta_j) r'_b
        tmem_st16(s_taddr + 32 * (j - 1), T);
        tmem_wait_st();
        float sn, cs;
        sincospif(__fdiv_rn((float)(2 * ph), (float)FN), &sn, &cs);
        const float2 w = make_float2(cs, sn);
#pragma unroll
        for (int n2 = 0; n2 < 16; n2++) T[n2] = cfma(acc[n2], w, T[n2]);
    }
    if (j == M - 1) {   // end of the group: best data-bit hypothesis per lag
        float pg[16];
#pragma unroll
        for (int n2 = 0; n2 < 16; n2++) pg[n2] = cpower(T[n2]);
        for (int e = 1; e < M; e++) {
            float2 S[16];
            tmem_ld16(s_taddr + 32 * (e - 1), S);
            tmem_wait_ld();
#pragma unroll
            for (int n2 = 0; n2 < 16; n2++)
                pg[n2] = fmaxf(pg[n2], cpower(make_float2(2.0f * S[n2].x - T[n2].x, 2.0f * S[n2].y - T[n2].y)));
        }
#pragma unroll
        for (int n2 = 0; n2 < 16; n2++) P[n2] = (b == M - 1) ? pg[n2] : (P[n2] + pg[n2]);
        j = 0;
        ph = 0;
    } else {
        j++;
        ph += step;
        if (ph >= FN) ph -= FN;
    }
}

template <class PA, bool E1B>
__global__ void __launch_bounds__(256, E1B || PA::kCoh ? 1 : 2) k_profile(const PA p)
{
    extern __shared__ __align__(1024) unsigned char smem[];
    constexpr int L = E1B ? ACQ_LAGS_E1B : ACQ_LAGS_L1;
    constexpr int kTmemCols = E1B ? kE1bTmemCols : (PA::kCoh ? 2 * kCohPrefixCols : 0);
    const int row = blockIdx.x, t = threadIdx.x;
    const int slot = row % p.n_slots, cap = row / p.n_slots;
    if (!PA::kCoh && (p.sat_type[p.slot_sat[slot]] == ACQ_E1B) != E1B) return;   // a row of the other launch
    const acq_record rc = p.rec[row];
    const int marker = record_marker(rc, p.slot_sat, slot, p.sat_type, p.n_sats, p.dop_lo, p.dop_hi,
                                     (p.flags & ACQ_PROFILE_DETECTED) != 0, p.thr_l1, p.thr_e1b);
    float *prof = nullptr;
    if (p.profile) {
        if constexpr (PA::kCoh) {
            prof = p.profile + (size_t)row * L;
        } else {   // row offset: the L of every earlier slot of this capture (uniform loop: every thread counts)
            int e1b_before = 0;
            for (int s0 = 0; s0 < slot; s0 += 256) {
                const int s = s0 + t;
                e1b_before += __syncthreads_count(s < slot && p.sat_type[p.slot_sat[s]] == ACQ_E1B);
            }
            const size_t cap_len = (size_t)p.n_slots * ACQ_LAGS_L1 + (size_t)p.n_e1b_slots * (ACQ_LAGS_E1B - ACQ_LAGS_L1);
            prof = p.profile + (size_t)cap * cap_len + (size_t)slot * ACQ_LAGS_L1 + (size_t)e1b_before * (ACQ_LAGS_E1B - ACQ_LAGS_L1);
        }
    }
    if (marker != 0) {   // uniform: every thread read the same record
        const float nan = __int_as_float(0x7fc00000);   // quiet NaN
        if (t == 0) {
            acq_peak2 o;
            o.peak2 = o.ratio = o.noise_ex = nan;
            o.lag2 = marker;
            p.out[row] = o;
        }
        if (prof)
            for (int n = t; n < L; n += 256) prof[n] = nan;
        return;
    }
    const FftSmem3 s = fft_smem3_carve(smem);
    float *red_f = reinterpret_cast<float *>(smem + fft_smem3_bytes());   // [16] warp partials, [16] record's power, [48] TMEM slot
    int *red_i = reinterpret_cast<int *>(red_f + 32);                     // [8]
    float *pk = red_f + 16;
    float *Pt = reinterpret_cast<float *>(smem + fft_smem3_bytes() + kProfileRedBytes) + t;   // E1B, K > 1: [64][256]
    load_t2(s, p.tables, t);
    // this thread's TMEM: lane 32*(warp%4) + (t%32); E1B: columns [96*(warp/4), +96), [k2][n2] parked; coherent: columns
    // [kCohPrefixCols*(warp/4), +kCohPrefixCols), [s - 1][16 complex]
    uint32_t tmem_base = 0, taddr = 0;
    if constexpr (kTmemCols > 0) {
        tmem_base = tmem_alloc_cta<kTmemCols>(reinterpret_cast<uint32_t *>(red_f + 48), t);
        taddr = tmem_base + tmem_lane_base(t) + (uint32_t)((t >> 7) * (E1B ? 96 : kCohPrefixCols));
    }
    const float2 *base = p.tables + kT2Elems + t;
    int M = 1;
    if constexpr (PA::kCoh) M = p.m_coh;
    const int F = p.nvar, FN = F * kN;
    const int dop = code_row(p, rc.dop);
    const int v = rc.dop - F * dop;
    int step = (v * kN - 16 * dop * F) % FN;   // theta_j in units of 1 / (F N) cycle: j * step mod F N
    if (step < 0) step += FN;
    Peak best;
    best.p = -1.0f;   // every power (>= 0) wins over it
    best.n = 0x7fffffff;
    best.sum = 0.0f;
    int buf = 0, j = 0, ph = 0;
    float P[16];    // C/A: block (group) sums of this thread's lags lag_of3(t, n2)
    float2 T[16];   // C/A: the running group sum
    for (int b = 0; b < p.K; b++) {
        const int cshift = !PA::kCoh && p.n_shift > 1 ? code_shift(b, rc.dop, p.cd_div) : 0;
        const float2 *D = spectrum_row(p, cap, b, v, cshift);
        float2 x[16], acc[16];
#pragma unroll 1
        for (int k2 = 0; k2 < 4; k2++) {
            {   // x[a] = conj(data[k]) * code[k - dop], k = 1024 a + 4 t + k2   (search.cpp:471; load_products)
                const int r = (k2 - dop) & 3;
                const int q = (k2 - dop - r) >> 2;
                const float2 *Dk = D + k2 * kSub + t;
                const float2 *Ek = p.Ep + (size_t)(rc.sat * 4 + r) * p.ext_len + p.Q + q + t;
#pragma unroll
                for (int a = 0; a < 16; a++) x[a] = cmul_conj_a(__ldg(Dk + 256 * a), __ldg(Ek + 256 * a));
            }
            subfft4096_inv3(x, k2, __ldg(base + k2 * 256), buf, s, t);
            buf ^= 1;
            if constexpr (E1B) {
                if (k2 < 3) {
                    float2 z[16];
#pragma unroll
                    for (int n2 = 0; n2 < 16; n2++) z[n2] = (k2 == 0) ? x[r16(n2)] : cmul(x[r16(n2)], c_cC[k2][n2]);
                    tmem_st16(taddr + 32 * k2, z);
                    tmem_wait_st();
                }
            } else {   // lags 0..4095 only: m = 0 of the radix-4 combine, accumulated as in k_search_l1
                if (k2 == 0) {
#pragma unroll
                    for (int n2 = 0; n2 < 16; n2++) acc[n2] = x[r16(n2)];
                } else {
#pragma unroll
                    for (int n2 = 0; n2 < 16; n2++) acc[n2] = cfma(x[r16(n2)], c_cC[k2][n2], acc[n2]);
                }
            }
        }
        const bool last = b + 1 == p.K;
        if constexpr (E1B) {   // radix-4 combine over k2 (k_search_e1b / k_search_e1b_multi), lags lag_of3(t, n2) + 4096 m
#pragma unroll
            for (int c4 = 0; c4 < 4; c4++) {
                float2 za[4], zb[4], zc[4];
                tmem_ld4(taddr + 0 * 32 + 8 * c4, za);
                tmem_ld4(taddr + 1 * 32 + 8 * c4, zb);
                tmem_ld4(taddr + 2 * 32 + 8 * c4, zc);
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
                        float pw = cpower(zz[m]);
                        if (b > 0) pw = Pt[(4 * n2 + m) * 256] + pw;
                        if (!last) Pt[(4 * n2 + m) * 256] = pw;
                        const int n = lag_of3(t, n2) + 4096 * m;
                        if (last && n < L) profile_visit(n, pw, rc.lag, p.excl, L, best, pk, prof);
                    }
                }
            }
        } else {
            coh_fold(acc, T, P, j, ph, b, M, step, FN, taddr);
        }
    }
    if constexpr (!E1B) {
#pragma unroll
        for (int n2 = 0; n2 < 16; n2++) {
            const int n = lag_of3(t, n2);
            if (n < L) profile_visit(n, P[n2], rc.lag, p.excl, L, best, pk, prof);
        }
    }
    const Peak tot = block_reduce_peak(best, red_f, red_i, t);   // its barrier also publishes *pk
    if (t == 0) {
        acq_peak2 o;
        o.peak2 = tot.p;
        o.lag2 = tot.n;
        o.ratio = __fdiv_rn(*pk, tot.p);
        o.noise_ex = __fdiv_rn(tot.sum, (float)(L - 2 * p.excl - 1));
        p.out[row] = o;
    }
    if constexpr (kTmemCols > 0) tmem_free_cta<kTmemCols>(tmem_base, t);
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
#ifdef ACQ_VARIANT_E1B_LDG
static size_t search_e1b_ldg_smem_bytes() { return fft_smem3_bytes() + 64 * sizeof(float); }
#endif

// The search kernel of argument type PA for a launch of `kind` with K > 1 (multi) or K = 1, and its dynamic shared
// memory.  launch_search_as launches what it returns and configure_search_kernels configures what it returns for every
// (kind, multi), so every search kernel a launch can pick is configured.
template <class PA>
struct SearchKernel {
    void (*f)(PA);
    size_t smem;
};
template <class PA>
static SearchKernel<PA> search_kernel(int kind, bool multi)
{
    if constexpr (PA::kCoh) {
        return {k_search_l1_coh<PA>, l1_multi_smem_bytes()};
    } else {
        switch (kind) {
        case kSearchE1bCluster:
            return {multi ? k_search_e1b_cluster<true, PA> : k_search_e1b_cluster<false, PA>, search_e1b_cluster_smem_bytes()};
        case kSearchE1b:
            if (multi) return {k_search_e1b_multi<PA>, e1b_multi_smem_bytes()};
            return {k_search_e1b<PA>, search_e1b_smem_bytes()};
        case kSearchL1Multi: return {k_search_l1_multi<PA>, l1_multi_smem_bytes()};
        case kSearchL1Cr: return {k_search_l1_cr<PA>, l1_multi_smem_bytes()};
        default:
#ifdef ACQ_VARIANT_L1_MULTI_TW   // the K > 1 form that keeps the stage-B twiddles (not the code run) in tensor memory
            if constexpr (std::is_same_v<PA, SearchArgs>)
                if (multi) return {k_search_l1<true, PA>, search_l1_smem_bytes()};
#endif
            if (multi) return {k_search_l1_multi<PA>, l1_multi_smem_bytes()};
            return {k_search_l1<false, PA>, search_l1_smem_bytes()};
        }
    }
}

template <class PA>
static cudaError_t configure_search_kernels()
{
    cudaError_t e = cudaSuccess;
    for (int kind : {kSearchL1, kSearchL1Multi, kSearchL1Cr, kSearchE1b, kSearchE1bCluster})
        for (bool multi : {false, true}) {
            const SearchKernel<PA> k = search_kernel<PA>(kind, multi);
            if ((e = cudaFuncSetAttribute(k.f, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)k.smem)) ||
                (e = cudaFuncSetAttribute(k.f, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared)))
                return e;
        }
    return e;
}

cudaError_t search_kernels_configure()
{
    cudaError_t e;
    if ((e = configure_search_kernels<SearchArgs>()) || (e = configure_search_kernels<AidedSearchArgs>()) ||
        (e = configure_search_kernels<CohSearchArgs>()) || (e = configure_search_kernels<AidedCohSearchArgs>()))
        return e;
#ifdef ACQ_VARIANT_E1B_LDG
    if ((e = cudaFuncSetAttribute(k_search_e1b_ldg, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)search_e1b_ldg_smem_bytes())))
        return e;
#endif
    const int fw = (int)fwd_smem_bytes(), fc = (int)(fft_smem3_bytes() + 2 * sizeof(float2) * kSub);
    if ((e = cudaFuncSetAttribute(k_fwd_fft_cluster<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, fc))) return e;
    if ((e = cudaFuncSetAttribute(k_fwd_fft_cluster<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, fc))) return e;
    if ((e = cudaFuncSetAttribute(k_fwd_fft<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, fw))) return e;
    if ((e = cudaFuncSetAttribute(k_fwd_fft<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, fw))) return e;
    if ((e = cudaFuncSetAttribute(k_profile<ProfileArgs, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)profile_smem_bytes(false, 1)))) return e;
    if ((e = cudaFuncSetAttribute(k_profile<ProfileArgs, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)profile_smem_bytes(true, 2)))) return e;
    if ((e = cudaFuncSetAttribute(k_profile<ProfileCohArgs, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)profile_smem_bytes(false, 1)))) return e;
    // One shared-memory carveout for every kernel of a search.  Left to the driver, the C/A kernel (2 x 96.3 KiB) runs
    // its SMs at the 196 KiB split and the E1B kernel (2 x 103.8 KiB) at 228 KiB, and an SM changes its split only when
    // it is empty: in a GPS + Galileo search the E1B CTAs -- launched to move in as the C/A CTAs retire -- entered no SM
    // before BOTH its C/A CTAs had gone (trace: first E1B CTA at 54.8 us although half the C/A CTAs leave by 50 us).
    // (the search kernels: configure_search_kernels)
    const void *chain[] = {(const void *)k_front_end<false>, (const void *)k_front_end<true>, (const void *)k_front_end_arg,
                           (const void *)k_fwd_fft<true>, (const void *)k_fwd_fft<false>, (const void *)k_fwd_fft_cluster<true>,
                           (const void *)k_fwd_fft_cluster<false>, (const void *)k_coh_variants, (const void *)k_pick_small,
                           (const void *)k_best_dop};
    for (const void *f : chain)
        if ((e = cudaFuncSetAttribute(f, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared))) return e;
    return cudaSuccess;
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
// The K = 1 full-bin kernel for most of round 2 (one CTA per SM, two teams with staging warps, capture residue resident,
// contiguous team ranges; since removed, DESIGN.md section 4) was +4.7 % over k_search_l1<false> ON THE STATIC STRIDE
// (6.30 -> 6.02 ms, 128-capture farm).  Most of that turned out to be the static stride's own loss -- the two CTAs of an
// SM run at different rates (see claim_tile) -- which the two-team CTA happened not to have: with claimed tiles
// k_search_l1<false> does the same farm in 5.78 ms, the two-team kernel in 5.96 ms, and k_search_l1_cr -- the resident
// capture residue in the two-CTA form, residue loop fully unrolled at 126 registers -- in 5.24 ms (32.1 M tiles/s).  On
// the reference's one-capture search: 70.9 us through acq_search against 75.4 us (k_search_l1<false>) and 77.5 us (the
// two-team kernel).
#ifndef ACQ_FORCE_L1_CTA
#define ACQ_FORCE_L1_CTA 0   // variant l1_cta: always k_search_l1<false> for K = 1 (the kernel-equivalence tests)
#endif
int search_kind_l1(int K, int half_bin)
{
#ifdef ACQ_VARIANT_L1_MULTI_TW
    return kSearchL1;   // this experiment build runs every C/A search on k_search_l1<MULTI>
#endif
    if (K > 1) return kSearchL1Multi;
    if (half_bin || ACQ_FORCE_L1_CTA) return kSearchL1;
    // full bins: the capture-resident kernel (chunks claimed from six rounds of tiles per CTA up, static stride below)
    return kSearchL1Cr;
}

// Which E1B search kernel: the cluster/DSMEM form when every tile can have a cluster of its own (one wave: 9 us per tile
// against 12.5 us for the one-CTA form, measured).  With more tiles than that the one-CTA-per-tile forms (k_search_e1b,
// k_search_e1b_multi for non-coherent sums) have ~2.9x the throughput.
#ifndef ACQ_FORCE_E1B_KERNEL
#define ACQ_FORCE_E1B_KERNEL 0   // variants e1b_cta / e1b_cluster: 1 = always the one-CTA form, 2 = always the cluster form
#endif
int search_kind_e1b(long long n_tiles, int sm_count)
{
    if (ACQ_FORCE_E1B_KERNEL) return ACQ_FORCE_E1B_KERNEL == 2 ? kSearchE1bCluster : kSearchE1b;
    return n_tiles <= sm_count / 4 ? kSearchE1bCluster : kSearchE1b;
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
    if (kind == kSearchL1Coh) cap = sm_count;  // one per SM (512 tensor-memory columns each)
    return (int)(n_tiles < cap ? n_tiles : cap);
}

template <class PA>
static int launch_search_as(PA a, int kind, int sm_count, cudaStream_t st, bool pdl)
{
    const int grid = search_grid_ctas(a.n_tiles, kind, sm_count);
    if (grid <= 0) return 0;
    if (!search_claims_tiles(a.n_tiles, grid)) a.tile_ctr = nullptr;   // few rounds: static stride
    if (kind == kSearchL1Cr) search_chunks(a.n_tiles, 2 * sm_count, &a.ck_n16, &a.ck_n4);
    SearchKernel<PA> k = search_kernel<PA>(kind, a.K > 1);
#ifdef ACQ_VARIANT_E1B_LDG   // one-CTA E1B search with its operands straight from L2, full-range searches only
    if constexpr (std::is_same_v<PA, SearchArgs>)
        if (kind == kSearchE1b) k = {k_search_e1b_ldg, search_e1b_ldg_smem_bytes()};
#endif
    // the cluster form runs a cluster of four CTAs per tile
    launch_k(k.f, kind == kSearchE1bCluster ? 4 * grid : grid, 256, k.smem, st, pdl, a);
    return 1;
}

int launch_search(const SearchArgs &a, bool e1b, int sm_count, cudaStream_t st, bool pdl)
{
    const int kind = e1b ? search_kind_e1b(a.n_tiles, sm_count) : search_kind_l1(a.K, a.half_bin);
    if (a.dop_center) return launch_search_as(AidedSearchArgs(a), kind, sm_count, st, pdl);
    return launch_search_as(a, kind, sm_count, st, pdl);
}

int launch_search_coh(const CohSearchArgs &a, int sm_count, cudaStream_t st, bool pdl)
{
    if (a.dop_center) return launch_search_as(AidedCohSearchArgs(a), kSearchL1Coh, sm_count, st, pdl);
    return launch_search_as(a, kSearchL1Coh, sm_count, st, pdl);
}

int launch_coh_variants(float2 *x2, const float2 *rot, int n_rows, int F, int K, cudaStream_t st)
{
    int launched = 0;
    for (int r0 = 0; r0 < n_rows; r0 += 32768) {  // gridDim.y <= 65535
        const int nr = (n_rows - r0 < 32768) ? (n_rows - r0) : 32768;
        k_coh_variants<<<dim3(kN / 256, nr), 256, 0, st>>>(x2 + (size_t)r0 * F * kN, rot, F, K, r0);
        launched++;
    }
    return launched;
}

template <class RA>
int launch_refine(const RA &a, int n_rows, cudaStream_t st)
{
    if (n_rows <= 0) return 0;
    k_refine<RA><<<n_rows, 256, 0, st>>>(a);
    return 1;
}
template int launch_refine(const RefineArgs &, int, cudaStream_t);
template int launch_refine(const RefineCohArgs &, int, cudaStream_t);

template <class PA>
int launch_profile(const PA &a, int n_rows, cudaStream_t st)
{
    if (n_rows <= 0) return 0;
    int n = 0;
    if (a.n_slots > a.n_e1b_slots) {
        k_profile<PA, false><<<n_rows, 256, profile_smem_bytes(false, a.K), st>>>(a);
        n++;
    }
    if constexpr (!PA::kCoh) {
        if (a.n_e1b_slots > 0) {
            k_profile<PA, true><<<n_rows, 256, profile_smem_bytes(true, a.K), st>>>(a);
            n++;
        }
    }
    return n;
}
template int launch_profile(const ProfileArgs &, int, cudaStream_t);
template int launch_profile(const ProfileCohArgs &, int, cudaStream_t);

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
