// acq_fft.cuh -- register/shared-memory FFT building blocks for the acquisition kernels (sm_100a).
//
// The 16384-point inverse transform of the correlator (reference gps/search.cpp:241,481:
// fftwf BACKWARD, unnormalised, e^{+j2*pi*k*n/N}) is decomposed as
//
//     k = 1024*a + 64*b + 4*c + k2        n = n0 + 16*n1 + 256*n2 + 4096*m
//     (a,b,c,n0,n1,n2 in 0..15;  k2,m in 0..3)
//
//     W^{kn} = W16^{a n0} . W256^{b n0} W16^{b n1} . W16384^{(4c+k2)(n0+16 n1)} W64^{(4c+k2) n2} . i^{k2 m}
//
// i.e. for each input residue k2 (a "polyphase" quarter of the spectrum, contiguous in the
// polyphase HBM layout) one 4096-point sub-FFT made of three radix-16 passes held in registers
// (stage A over a, stage B over b, stage C over c) with two shared-memory exchanges, followed by
// a radix-4 combine over k2 that lives in registers.  The C/A search only needs the first 4092
// lags (m = 0), so its combine is a plain accumulation and three quarters of the last radix-4
// are never computed.
//
// 256 threads, 16 points per thread.  Thread roles:
//   stage A: t = 16*b + c    holds a = 0..15      -> outputs n0
//   stage B: t = 16*n0 + c   holds b = 0..15      -> outputs n1
//   stage C: t = 16*n0 + n1  holds c = 0..15      -> outputs n2   (lag n = (t>>4) + 16*(t&15) + 256*n2 + 4096*m)
//
// Twiddles: stage A multiplies output n0 by W16384^{(4t+k2)*n0} = b^{n0}, successive powers of one
// per-thread base b (table of 4 x 256 bases in global memory, computed on the host in double
// precision); stage B uses W1024^{(4c+k2)*n1} (7.5 KiB shared table); stage C's W64^{k2*n2} are constants.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "acq_geom.h"

namespace acq {

// Constant twiddles (filled by the host at engine creation; identical on every device).
//   c_cC[k2][n2] = W64^{k2*n2}      (e^{+j...}: inverse transform)
// Defined here (not extern): this header is included by exactly one translation unit
// (acq_kernels.cu), so no relocatable device code is needed.
__constant__ float2 c_cC[4][16];

// ---------------------------------------------------------------------------------------------
// complex helpers
// ---------------------------------------------------------------------------------------------
// Complex arithmetic on packed f32x2 instructions (sm_100 FADD2 / FMUL2 / FFMA2).  A complex value is one
// aligned register pair (re, im).  The packed instructions carry free operand modifiers -- lane swap
// (.LO_HI), negate one lane (.NP), negate both (-R) -- and take a scalar register as a broadcast operand
// (R.F32), so  a +- b,  a +- j*b  are ONE instruction and a complex multiply is TWO (FMUL2 + FFMA2).  The FMA
// pipe does the same work as with scalar instructions; the gain is issue slots (half as many FP
// instructions) and no register shuffling.
__device__ __forceinline__ float2 bc(float s) { return make_float2(s, s); }              // R.F32 broadcast
__device__ __forceinline__ float2 jmul(float2 a) { return make_float2(-a.y, a.x); }     // j*a  (-R.LO_HI.NP)
__device__ __forceinline__ float2 cneg(float2 a) { return make_float2(-a.x, -a.y); }
__device__ __forceinline__ float2 cadd(float2 a, float2 b) { return __fadd2_rn(a, b); }
__device__ __forceinline__ float2 csub(float2 a, float2 b) { return __fadd2_rn(a, cneg(b)); }
__device__ __forceinline__ float2 cadd_jb(float2 a, float2 b) { return __fadd2_rn(a, jmul(b)); }        // a + j*b
__device__ __forceinline__ float2 csub_jb(float2 a, float2 b) { return __fadd2_rn(a, cneg(jmul(b))); }  // a - j*b
// a * w = a*w.x + (j*a)*w.y
__device__ __forceinline__ float2 cmul(float2 a, float2 w)
{
    return __ffma2_rn(jmul(a), bc(w.y), __fmul2_rn(a, bc(w.x)));
}
// c + a * w
__device__ __forceinline__ float2 cfma(float2 a, float2 w, float2 c)
{
    return __ffma2_rn(jmul(a), bc(w.y), __ffma2_rn(a, bc(w.x), c));
}
// conj(a) * b  (reference support/simd.cpp:12-40: re = ar*br + ai*bi, im = ar*bi - ai*br) = b*a.x - (j*b)*a.y
__device__ __forceinline__ float2 cmul_conj_a(float2 a, float2 b)
{
    return __ffma2_rn(cneg(jmul(b)), bc(a.y), __fmul2_rn(b, bc(a.x)));
}
__device__ __forceinline__ float2 mul_pj(float2 a) { return jmul(a); }        // * (+j)
__device__ __forceinline__ float2 mul_mj(float2 a) { return cneg(jmul(a)); }  // * (-j)

// Inverse radix-4 butterfly (W4 = +j), in place on four registers.
__device__ __forceinline__ void radix4_inv(float2 &a, float2 &b, float2 &c, float2 &d)
{
    const float2 apc = cadd(a, c), amc = csub(a, c);
    const float2 bpd = cadd(b, d), bmd = csub(b, d);
    a = cadd(apc, bpd);
    b = cadd_jb(amc, bmd);
    c = csub(apc, bpd);
    d = csub_jb(amc, bmd);
}

// Inverse 16-point DFT in registers: X[n] = sum_a x[a] e^{+2*pi*j*a*n/16}.
// Input x[a] in natural order.  Output X[n] is left at register index  r16(n) = (n >> 2) | ((n & 3) << 2).
__host__ __device__ constexpr int r16(int n) { return (n >> 2) | ((n & 3) << 2); }

__device__ __forceinline__ void radix16_inv(float2 (&x)[16])
{
    constexpr float C1 = 0.92387953251128675613f;  // cos(pi/8)
    constexpr float S1 = 0.38268343236508977173f;  // sin(pi/8)
    constexpr float R2 = 0.70710678118654752440f;  // sqrt(1/2)
    // layer 1: for each a0, radix-4 over a = a0 + 4*a1  ->  u[a0][nl] at index a0 + 4*nl
#pragma unroll
    for (int a0 = 0; a0 < 4; a0++) radix4_inv(x[a0], x[a0 + 4], x[a0 + 8], x[a0 + 12]);
    // Twiddles u[a0][nl] *= W16^{a0*nl} folded into layer 2 where they are (+-1 +- j)/sqrt2: the 1/sqrt2 rides
    // on the fused multiply-add of the following butterfly (4 packed instructions fewer than twiddle-then-add).
    // nl = 0: no twiddles
    radix4_inv(x[0], x[1], x[2], x[3]);
    {   // nl = 1: b = x5 W^1, c = x6 W^2 = R2 (x6 + j x6), d = x7 W^3
        const float2 s6 = cadd(x[6], jmul(x[6]));
        const float2 b = cmul(x[5], make_float2(C1, S1)), d = cmul(x[7], make_float2(S1, C1));
        const float2 apc = __ffma2_rn(s6, bc(R2), x[4]), amc = __ffma2_rn(s6, bc(-R2), x[4]);
        const float2 bpd = cadd(b, d), bmd = csub(b, d);
        x[4] = cadd(apc, bpd);
        x[5] = cadd_jb(amc, bmd);
        x[6] = csub(apc, bpd);
        x[7] = csub_jb(amc, bmd);
    }
    {   // nl = 2: b = x9 W^2 = R2 (x9 + j x9), c = j x10, d = x11 W^6 = R2 (j x11 - x11)
        const float2 s9 = cadd(x[9], jmul(x[9])), s11 = csub(jmul(x[11]), x[11]);
        const float2 apc = cadd_jb(x[8], x[10]), amc = csub_jb(x[8], x[10]);
        const float2 bpd = cadd(s9, s11), bmd = csub(s9, s11);  // both still to be scaled by R2
        x[8] = __ffma2_rn(bpd, bc(R2), apc);
        x[9] = __ffma2_rn(jmul(bmd), bc(R2), amc);
        x[10] = __ffma2_rn(bpd, bc(-R2), apc);
        x[11] = __ffma2_rn(jmul(bmd), bc(-R2), amc);
    }
    {   // nl = 3: b = x13 W^3, c = x14 W^6 = R2 (j x14 - x14), d = x15 W^9
        const float2 s14 = csub(jmul(x[14]), x[14]);
        const float2 b = cmul(x[13], make_float2(S1, C1)), d = cmul(x[15], make_float2(-C1, -S1));
        const float2 apc = __ffma2_rn(s14, bc(R2), x[12]), amc = __ffma2_rn(s14, bc(-R2), x[12]);
        const float2 bpd = cadd(b, d), bmd = csub(b, d);
        x[12] = cadd(apc, bpd);
        x[13] = cadd_jb(amc, bmd);
        x[14] = csub(apc, bpd);
        x[15] = csub_jb(amc, bmd);
    }
}

// ---------------------------------------------------------------------------------------------
// Tensor memory (TMEM) as thread-private storage: tcgen05.st / tcgen05.ld with the .32x32b shape map thread i
// of a warp to TMEM lane 32*(warp%4)+i and N consecutive 32-bit columns to N registers.  Data parked there
// moves over the tensor-memory datapath, not the L1/shared data pipe.  taddr = (lane base << 16) | column.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const float2 (&v)[16])
{
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,"
        "%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31,%32};" ::"r"(taddr),
        "f"(v[0].x), "f"(v[0].y), "f"(v[1].x), "f"(v[1].y), "f"(v[2].x), "f"(v[2].y), "f"(v[3].x), "f"(v[3].y), "f"(v[4].x),
        "f"(v[4].y), "f"(v[5].x), "f"(v[5].y), "f"(v[6].x), "f"(v[6].y), "f"(v[7].x), "f"(v[7].y), "f"(v[8].x), "f"(v[8].y),
        "f"(v[9].x), "f"(v[9].y), "f"(v[10].x), "f"(v[10].y), "f"(v[11].x), "f"(v[11].y), "f"(v[12].x), "f"(v[12].y),
        "f"(v[13].x), "f"(v[13].y), "f"(v[14].x), "f"(v[14].y), "f"(v[15].x), "f"(v[15].y)
        : "memory");
}
__device__ __forceinline__ void tmem_ld4(uint32_t taddr, float2 (&v)[4])
{
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=f"(v[0].x), "=f"(v[0].y), "=f"(v[1].x), "=f"(v[1].y), "=f"(v[2].x), "=f"(v[2].y), "=f"(v[3].x),
                   "=f"(v[3].y)
                 : "r"(taddr)
                 : "memory");
}
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

__device__ __forceinline__ void tmem_st8(uint32_t taddr, const float2 (&v)[8])
{
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};" ::"r"(taddr),
        "f"(v[0].x), "f"(v[0].y), "f"(v[1].x), "f"(v[1].y), "f"(v[2].x), "f"(v[2].y), "f"(v[3].x), "f"(v[3].y), "f"(v[4].x),
        "f"(v[4].y), "f"(v[5].x), "f"(v[5].y), "f"(v[6].x), "f"(v[6].y), "f"(v[7].x), "f"(v[7].y)
        : "memory");
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, float2 (&v)[8])
{
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
        : "=f"(v[0].x), "=f"(v[0].y), "=f"(v[1].x), "=f"(v[1].y), "=f"(v[2].x), "=f"(v[2].y), "=f"(v[3].x), "=f"(v[3].y),
          "=f"(v[4].x), "=f"(v[4].y), "=f"(v[5].x), "=f"(v[5].y), "=f"(v[6].x), "=f"(v[6].y), "=f"(v[7].x), "=f"(v[7].y)
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float2 (&v)[16])
{
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
        "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
        : "=f"(v[0].x), "=f"(v[0].y), "=f"(v[1].x), "=f"(v[1].y), "=f"(v[2].x), "=f"(v[2].y), "=f"(v[3].x), "=f"(v[3].y),
          "=f"(v[4].x), "=f"(v[4].y), "=f"(v[5].x), "=f"(v[5].y), "=f"(v[6].x), "=f"(v[6].y), "=f"(v[7].x), "=f"(v[7].y),
          "=f"(v[8].x), "=f"(v[8].y), "=f"(v[9].x), "=f"(v[9].y), "=f"(v[10].x), "=f"(v[10].y), "=f"(v[11].x), "=f"(v[11].y),
          "=f"(v[12].x), "=f"(v[12].y), "=f"(v[13].x), "=f"(v[13].y), "=f"(v[14].x), "=f"(v[14].y), "=f"(v[15].x), "=f"(v[15].y)
        : "r"(taddr)
        : "memory");
}
// One warp allocates `cols` columns (power of two >= 32) for the CTA; every thread gets the base address.
// Contains a __syncthreads().
template <int COLS>
__device__ __forceinline__ uint32_t tmem_alloc_cta(uint32_t *slot, int t)
{
    if ((t >> 5) == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                         (uint32_t)__cvta_generic_to_shared(slot)),
                     "n"(COLS)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    return *slot;
}
template <int COLS>
__device__ __forceinline__ void tmem_free_cta(uint32_t base, int t)
{
    __syncthreads();
    if ((t >> 5) == 0)
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(base), "n"(COLS) : "memory");
}
// lane base of this thread's warp (bits 31:16 of a TMEM address)
__device__ __forceinline__ uint32_t tmem_lane_base(int t) { return (uint32_t)(((t >> 5) & 3) * 32) << 16; }

// ---------------------------------------------------------------------------------------------
// The 4096-point sub-FFT of one input residue k2.
//   * The stage-A twiddles W16384^{(4t+k2)*n0}, n0 = 1..15, are successive powers of ONE per-thread base
//     b = W16384^{4t+k2}: a chain of packed complex multiplies instead of a 30 KiB shared-memory table
//     read once per sub-FFT.  The FMA pipe does about the same work as the table fix-ups it replaces; the
//     L1/shared data pipe -- the busiest unit of the search kernel (profiles/) -- moves 30 KiB less per
//     sub-FFT.  Worst-case twiddle error grows to ~15 ulp-of-1 (1e-6), far inside the
//     1e-3 budget; tests/test_gpu_parity.py checks spectra to 1e-5.
//   * The A->B exchange buffer S1 is double buffered (successive sub-FFTs alternate), and the B->C
//     exchange is private to each half-warp: with stage-B thread t = 16*n0 + c and stage-C thread
//     t = 16*n0 + n1, the 16 threads sharing n0 transpose a 16x16 tile among themselves, so a
//     __syncwarp() replaces the second CTA barrier.  One __syncthreads() per sub-FFT remains:
//     writes A(i+1) go to the buffer last read in B(i-1), and every warp passed barrier(i) only after
//     finishing its B(i-1) reads.
// Stage-C thread t then owns lags n = (t >> 4) + 16*(t & 15) + 256*n2.
// ---------------------------------------------------------------------------------------------
// Stage-A output twiddles W16384^{(4t+k2) n0} = b^{n0}, n0 = 1..15, as ACQ_TW_CHAINS interleaved chains of powers
// (chain i holds b^{i+1}, b^{i+1+C}, ...; every chain advances by b^C): always 14 complex multiplies, dependent
// depth 14 with one chain, 8 with two, 6 with four (measured: two chains +0.5 % on cfg2/cfg5, +0.9 % on cfg3 over one;
// four no better).  dst[n0 * STRIDE] = x[r16(n0)] * b^{n0}.
#ifndef ACQ_TW_CHAINS
#define ACQ_TW_CHAINS 2
#endif
template <int STRIDE>
__device__ __forceinline__ void stage_a_store(const float2 (&x)[16], const float2 b, float2 *dst)
{
    constexpr int C = ACQ_TW_CHAINS;
    float2 tw[C];
    tw[0] = b;
#pragma unroll
    for (int i = 1; i < C; i++) tw[i] = cmul(tw[i - 1], b);
    const float2 step = tw[C - 1];
    dst[0] = x[r16(0)];
#pragma unroll
    for (int n0 = 1; n0 < 16; n0++) {
        const int i = (n0 - 1) % C;
        dst[n0 * STRIDE] = cmul(x[r16(n0)], tw[i]);
        if (n0 + C <= 15) tw[i] = cmul(tw[i], step);
    }
}

constexpr int kS2TileElems = 16 * 17;  // one padded 16x16 tile per half-warp

struct FftSmem3 {
    float2 *T2;  // [4][15][16]
    float2 *S1;  // [2][4096]
    float2 *S2;  // [16 half-warps][16*17]
};

__host__ __device__ constexpr size_t fft_smem3_bytes()
{
    return sizeof(float2) * (size_t)(kT2Elems + 2 * kS1Elems + 16 * kS2TileElems);
}

__device__ __forceinline__ FftSmem3 fft_smem3_carve(unsigned char *base)
{
    FftSmem3 s;
    s.T2 = reinterpret_cast<float2 *>(base);
    s.S1 = s.T2 + kT2Elems;
    s.S2 = s.S1 + 2 * kS1Elems;
    return s;
}

__device__ __forceinline__ int lag_of3(int t, int n2) { return (t >> 4) + 16 * (t & 15) + 256 * n2; }

//   in : x[a] = input element k = 1024*a + 4*t + k2;  b = W16384^{4t+k2};  buf = parity of the sub-FFT count
//   out: x[r16(n2)] = stage-C output for lag lag_of3(t, n2), before the W64^{k2*n2} factor
__device__ __forceinline__ void subfft4096_inv3(float2 (&x)[16], const int k2, const float2 b, const int buf,
                                                const FftSmem3 &s, const int t)
{
    radix16_inv(x);
    stage_a_store<256>(x, b, s.S1 + buf * kS1Elems + t);
    // stage-B twiddles W1024^{(4c+k2)*n1} do not depend on the exchange: first batch before the barrier
    float2 tw[8];
    const float2 *twp = s.T2 + k2 * (15 * 16) + (t & 15);
#pragma unroll
    for (int i = 0; i < 8; i++) tw[i] = twp[i * 16];  // n1 = 1..8
    __syncthreads();
    // ---- stage B: thread (n0, c) = (t >> 4, t & 15) gathers b = 0..15
    {
        const float2 *src = s.S1 + buf * kS1Elems + (t & ~15) * 16 + (t & 15);
#pragma unroll
        for (int bb = 0; bb < 16; bb++) x[bb] = src[16 * bb];
    }
    radix16_inv(x);
    float2 *tile = s.S2 + (t >> 4) * kS2TileElems;
    {
        float2 *dst = tile + (t & 15);  // element (n1, c) at n1*17 + c
        dst[0] = x[r16(0)];
#pragma unroll
        for (int i = 0; i < 8; i++) dst[(i + 1) * 17] = cmul(x[r16(i + 1)], tw[i]);
#pragma unroll
        for (int i = 0; i < 7; i++) tw[i] = twp[(i + 8) * 16];  // n1 = 9..15
#pragma unroll
        for (int i = 0; i < 7; i++) dst[(i + 9) * 17] = cmul(x[r16(i + 9)], tw[i]);
    }
    __syncwarp();
    // ---- stage C: thread (n0, n1) = (t >> 4, t & 15) gathers c = 0..15
    {
        const float2 *src = tile + 17 * (t & 15);
#pragma unroll
        for (int c = 0; c < 16; c++) x[c] = src[c];
    }
    radix16_inv(x);
}

constexpr int kTwCols = 4 * 32;  // TMEM columns of one thread's stage-B twiddles (subfft4_park_twiddles)

// ---------------------------------------------------------------------------------------------
// Operand-prefetching form of the sub-FFT (used by k_search_l1).
//   * Both operands of the NEXT sub-FFT are staged by TMA bulk copies (cp.async.bulk + mbarrier complete_tx)
//     while the current one computes: the capture-spectrum residue D (32 KiB, contiguous in the polyphase
//     layout; one 2 KiB copy per exchange row) lands in the idle half of the double-buffered A->B exchange
//     buffer, exactly where thread t later writes its own stage-A outputs (it reads D[256 a + t] from row a,
//     column t and writes its output n0 to row n0, column t: the same 16 slots, so the reuse is
//     thread-private), and the code-spectrum run E (32 KiB + 16 B: the Doppler offset is only 8-byte aligned)
//     lands in a buffer of its own.  The L2 round trip leaves the dependent chain of every warp.
//   * The B->C tile of a half-warp lives in the exchange row that half-warp has just consumed (row n0, read by
//     nobody else), XOR-swizzled in 16-byte chunks -- conflict-free column writes and 128-bit row reads, no padding
//     (so a capture residue can still land in the buffer by one 32 KiB bulk copy) and no separate tile buffer.
//   * TMEM column 30/31 of residue k2 (the unused sixteenth twiddle slot) carries the stage-A base
//     W16384^{4t + (k2+1 mod 4)} of the NEXT sub-FFT, so it arrives with the stage-B twiddles.
// Shared memory per CTA: 2 x 34 KiB (S1) + 32 KiB + 16 B (E) + one mbarrier.
// ---------------------------------------------------------------------------------------------
constexpr int kEBufElems = kSub + 2;
constexpr int kRowElems = 256;                // exchange row; the B->C tile of a half-warp lives in it, XOR-swizzled
constexpr int kS1pElems = 16 * kRowElems;     // one half of the exchange buffer
struct FftSmem4 {
    float2 *S1;  // [2][16][256]
    float2 *E;   // [4098]
    unsigned long long *bar;
};
__host__ __device__ constexpr size_t fft_smem4_bytes() { return sizeof(float2) * (size_t)(2 * kS1pElems + kEBufElems) + 16; }
__device__ __forceinline__ FftSmem4 fft_smem4_carve(unsigned char *base)
{
    FftSmem4 s;
    s.S1 = reinterpret_cast<float2 *>(base);
    s.E = s.S1 + 2 * kS1pElems;
    s.bar = reinterpret_cast<unsigned long long *>(s.E + kEBufElems);
    return s;
}

// Programmatic dependent launch (PDL): the kernels of one search are launched back to back with
// cudaLaunchAttributeProgrammaticStreamSerialization, so a kernel's CTAs become resident and run their prologue
// (tensor-memory allocation, twiddle parking, barrier init -- nothing that reads or writes search data) while its
// predecessor drains.  pdl_wait() returns once every prerequisite grid has completed and its writes are visible;
// every thread of every kernel in the chain calls it before touching search data, so completion is transitive.
// Both are no-ops for a kernel launched without the attribute.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// Timeline instrumentation of the experiment variant "trace" (tools/trace_timeline.py): thread 0 of every CTA stamps
// %globaltimer at entry, after its wait for the preceding grid and at exit.  Compiled out of the product.
#ifdef ACQ_TRACE
constexpr int kTraceKernels = 6, kTraceCtas = 1024;
enum { kTrFrontEnd = 0, kTrFwdFft = 1, kTrSearchL1 = 2, kTrSearchE1b = 3, kTrPick = 4, kTrE1bCluster = 5 };
__device__ unsigned long long g_trace[kTraceKernels][kTraceCtas][4];
__device__ __forceinline__ void trace_stamp(int kernel, int slot)
{
    const unsigned cta = blockIdx.x + gridDim.x * blockIdx.y;
    if (threadIdx.x == 0 && cta < (unsigned)kTraceCtas) {
        unsigned long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        g_trace[kernel][cta][slot] = t;
    }
}
#define ACQ_TRACE_STAMP(kernel, slot) trace_stamp(kernel, slot)
#else
#define ACQ_TRACE_STAMP(kernel, slot)
#endif

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity)
{
    uint32_t ok;
    do {
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
            "selp.u32 %0, 1, 0, p;\n"
            "}\n"
            : "=r"(ok)
            : "r"(bar), "r"(parity)
            : "memory");
    } while (!ok);
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_load_1d(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
                 "l"(src), "r"(bytes), "r"(bar)
                 : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// Twiddle parking for subfft4096_inv4: this thread's stage-B twiddles (c = t & 15) to TMEM columns
// [32*k2 + 2*(n1-1), +2), plus the next residue's stage-A base in the sixteenth slot.  tables: T2 [4][15][16], then
// bases [4][256].
__device__ __forceinline__ void subfft4_park_twiddles(const float2 *__restrict__ tables, uint32_t tw_taddr, int t)
{
#pragma unroll
    for (int k2 = 0; k2 < 4; k2++) {
        float2 v[8];
#pragma unroll
        for (int h = 0; h < 2; h++) {
#pragma unroll
            for (int i = 0; i < 8; i++) {
                const int n1 = 8 * h + i + 1;
                v[i] = (n1 < 16) ? __ldg(tables + (k2 * 15 + (n1 - 1)) * 16 + (t & 15))
                                 : __ldg(tables + kT2Elems + ((k2 + 1) & 3) * 256 + t);
            }
            tmem_st8(tw_taddr + 32 * k2 + 16 * h, v);
        }
    }
    tmem_wait_st();
}

//   in : x[a] = product for input element k = 1024*a + 4*t + k2;  b = W16384^{4t+k2} (in/out: replaced by the
//        next residue's base);  S1b = this sub-FFT's half of S1
//   post_barrier(): called by every thread right after the CTA barrier (warp 0 issues the next TMA there)
//   out: x[r16(n2)] = stage-C output for lag lag_of3(t, n2), before the W64^{k2*n2} factor
// The B->C tile is swizzled in 16-byte chunks and read with 128-bit loads (below).  Measured against an 8-byte
// swizzle read with 64-bit loads (same box): +1.2 % on the K > 1 kernel (cfg2), +0.9 % on E1B (cfg3); on the K = 1
// kernel -0.8 % with the rolled residue loop, +1.5 % (cfg5) once that loop is unrolled by two.
template <class PostBarrier>
__device__ __forceinline__ void subfft4096_inv4(float2 (&x)[16], const int k2, float2 &b, float2 *S1b, const int t,
                                                const uint32_t tw_taddr, PostBarrier &&post_barrier)
{
    radix16_inv(x);
    stage_a_store<kRowElems>(x, b, S1b + t);
    float2 tw[8], tw2[8];
    tmem_ld8(tw_taddr + 32 * k2, tw);        // n1 = 1..8, in flight across the barrier
    tmem_ld8(tw_taddr + 32 * k2 + 16, tw2);  // n1 = 9..15, then the next residue's stage-A base
#define TW_AT(i) ((i) < 8 ? tw[(i)] : tw2[(i) - 8])
    __syncthreads();
    post_barrier();
    float2 *row = S1b + (t >> 4) * kRowElems;  // row n0 = t >> 4
    const int c = t & 15;
    {
        const float2 *src = row + c;
#pragma unroll
        for (int bb = 0; bb < 16; bb++) x[bb] = src[16 * bb];
    }
    radix16_inv(x);
    tmem_wait_ld();
    b = TW_AT(15);
    __syncwarp();  // the half-warp has consumed its row: reuse it as the B->C tile, element (n1, c) at 17 n1 + c
    {   // unpadded row, swizzled in 16-byte chunks: element (n1, c) in chunk (c >> 1) ^ (n1 & 7), slot c & 1 of tile row
        // n1, so that stage C reads two adjacent elements with one 128-bit load (half the loads and address XORs):
        // address = ((row + 8 c) ^ (16 (n1 & 7))) + 128 n1
        const uint32_t wb = smem_u32(row + c);
        asm volatile("st.shared.v2.f32 [%0], {%1, %2};" ::"r"(wb), "f"(x[r16(0)].x), "f"(x[r16(0)].y) : "memory");
#pragma unroll
        for (int i = 0; i < 15; i++) {
            const int n1 = i + 1;
            const float2 v = cmul(x[r16(n1)], TW_AT(i));
            asm volatile("st.shared.v2.f32 [%0], {%1, %2};" ::"r"((wb ^ (16u * (n1 & 7))) + 128u * n1), "f"(v.x), "f"(v.y) : "memory");
        }
    }
    __syncwarp();
    {   // this thread is now (n0, n1 = c): elements (c, 2 j), (c, 2 j + 1) in chunk j ^ (c & 7) of tile row c
        const uint32_t rb = smem_u32(row + 16 * c + 2 * (c & 7));
#pragma unroll
        for (int j = 0; j < 8; j++)
            asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];"
                         : "=f"(x[2 * j].x), "=f"(x[2 * j].y), "=f"(x[2 * j + 1].x), "=f"(x[2 * j + 1].y)
                         : "r"(rb ^ (16u * j))
                         : "memory");
    }
    radix16_inv(x);
}
#undef TW_AT

// Form of subfft4096_inv4 for kernels whose tensor memory is taken by parked data (k_search_e1b: 96 of a thread's
// 128 columns hold three residues): the stage-B twiddles W1024^{(4c+k2)*n1} come from a 7.5 KiB shared-memory
// table T2s (read before the barrier / during stage B, broadcast between the two half-warps), the stage-A base
// of the next residue from two TMEM columns at base_taddr + 2*((k2+1)&3).  Operand staging, exchange rows and
// the B->C swizzle are those of subfft4096_inv4.
__device__ __forceinline__ void tmem_ld1(uint32_t taddr, float2 &v)
{
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x2.b32 {%0,%1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_st1(uint32_t taddr, const float2 v)
{
    asm volatile("tcgen05.st.sync.aligned.32x32b.x2.b32 [%0], {%1,%2};" ::"r"(taddr), "f"(v.x), "f"(v.y) : "memory");
}

// Where the stage-A base W16384^{4t + k2'} of the NEXT residue k2' = (k2 + 1) & 3 comes from: two TMEM columns per
// residue (kernels with columns to spare), or the 8 KiB table in global memory (L1/L2-resident; kernels whose tensor
// memory is full).  issue() runs before the CTA barrier, get() after stage B: the latency is hidden either way.
struct BaseFromTmem {
    uint32_t taddr;  // columns [taddr + 2 k2', +2)
    float2 v;
    __device__ __forceinline__ void issue(int k2) { tmem_ld1(taddr + 2 * ((k2 + 1) & 3), v); }
    __device__ __forceinline__ float2 get()
    {
        tmem_wait_ld();
        return v;
    }
};
struct BaseFromGlobal {
    const float2 *bases;  // this thread's column of the [4][256] table: bases[256 k2']
    float2 v;
    __device__ __forceinline__ void issue(int k2) { v = __ldg(bases + 256 * ((k2 + 1) & 3)); }
    __device__ __forceinline__ float2 get() { return v; }
};

template <class BaseSrc, class PostBarrier>
__device__ __forceinline__ void subfft4096_inv4s(float2 (&x)[16], const int k2, float2 &b, float2 *S1b, const int t,
                                                 const float2 *T2s, BaseSrc base_src, PostBarrier &&post_barrier)
{
    radix16_inv(x);
    stage_a_store<256>(x, b, S1b + t);
    // all 15 stage-B twiddles before the barrier: with the residue loop of k_search_e1b unrolled 20.7 M tiles/s on
    // cfg3, against 20.35 M with eight before it and seven during stage B, and no spill
    float2 tw[15];
    const float2 *twp = T2s + k2 * (15 * 16) + (t & 15);
#pragma unroll
    for (int i = 0; i < 15; i++) tw[i] = twp[i * 16];  // n1 = 1..15
    base_src.issue(k2);
    __syncthreads();
    post_barrier();
    float2 *row = S1b + (t >> 4) * 256;  // row n0 = t >> 4
    const int c = t & 15;
    {
        const float2 *src = row + c;
#pragma unroll
        for (int bb = 0; bb < 16; bb++) x[bb] = src[16 * bb];
    }
    radix16_inv(x);
    b = base_src.get();
    __syncwarp();  // the half-warp has consumed its row: reuse it as the B->C tile, swizzled as in subfft4096_inv4
    {
        const uint32_t wb = smem_u32(row + c);
        asm volatile("st.shared.v2.f32 [%0], {%1, %2};" ::"r"(wb), "f"(x[r16(0)].x), "f"(x[r16(0)].y) : "memory");
#pragma unroll
        for (int i = 0; i < 8; i++) {
            const int n1 = i + 1;
            const float2 v = cmul(x[r16(n1)], tw[i]);
            asm volatile("st.shared.v2.f32 [%0], {%1, %2};" ::"r"((wb ^ (16u * (n1 & 7))) + 128u * n1), "f"(v.x), "f"(v.y) : "memory");
        }
#pragma unroll
        for (int i = 0; i < 7; i++) {
            const int n1 = i + 9;
            const float2 v = cmul(x[r16(n1)], tw[i + 8]);
            asm volatile("st.shared.v2.f32 [%0], {%1, %2};" ::"r"((wb ^ (16u * (n1 & 7))) + 128u * n1), "f"(v.x), "f"(v.y) : "memory");
        }
    }
    __syncwarp();
    {
        const uint32_t rb = smem_u32(row + 16 * c + 2 * (c & 7));
#pragma unroll
        for (int j = 0; j < 8; j++)
            asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];"
                         : "=f"(x[2 * j].x), "=f"(x[2 * j].y), "=f"(x[2 * j + 1].x), "=f"(x[2 * j + 1].y)
                         : "r"(rb ^ (16u * j))
                         : "memory");
    }
    radix16_inv(x);
}

}  // namespace acq
