// field.cuh — 256-bit Montgomery prime-field arithmetic for sm_100a on 8 x 32-bit limbs.
//
// Replaces what ark-ff's Fp256<MontBackend<_,4>> does for the reference's prover
// (reference call sites: src/backend/snark.rs:194,203-208 and everything inside
// Groth16::prove at snark.rs:364,442).  Same field, same Montgomery radix R = 2^256,
// values fully reduced, so canonical outputs are bit-identical.  (The G1 gather kernel's
// accumulator alone runs in a redundant form, [0, 2p), and is reduced before it is stored.)
//
// Multiplication is a CIOS Montgomery product built from carry-chained
// mad.lo.cc / madc.hi.cc rows; ptxas fuses each lo/hi pair into one
// IMAD.WIDE.U32(.X), so one product costs 128 wide multiply-adds + 8 IMADs on the
// fma pipe.  Two partial accumulators ("aligned" limbs k <-> column k, "offset"
// limbs k <-> column k+1) let every row be one uninterrupted carry chain.
//
// Every carry chain lives inside ONE asm statement, so the PTX condition-code
// register never has to survive between statements.  The same row primitives have
// a portable C++ body (used when this header is compiled for the host), which lets
// tests/test_field_host.py check the composition logic without a GPU.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define LZ_HD __host__ __device__ __forceinline__
#define LZ_COLD __host__ __device__ __noinline__
#else
#define LZ_HD inline
#define LZ_COLD inline
#endif
#define LZ_CONST_ARRAY(NAME, ...)                                   \
    LZ_HD static constexpr uint32_t NAME(int i) {                   \
        const uint32_t v[8] = {__VA_ARGS__};                        \
        return v[i];                                                \
    }

#include "bn254_constants.cuh"

namespace lzkp {

// --------------------------------------------------------------------------
// Row primitives.  D is an 8-limb accumulator; (s0..s3) are four multiplicand
// limbs, k the multiplier limb.  Pair t of D receives the 64-bit product s_t*k.
// --------------------------------------------------------------------------

// D = (s0,s1,s2,s3) * k
LZ_HD void row_mul(uint32_t (&D)[8], uint32_t s0, uint32_t s1, uint32_t s2, uint32_t s3, uint32_t k) {
    // 64-bit products: ptxas emits one IMAD.WIDE.U32 each.  (Written as mul.lo / mul.hi pairs it kept them apart as
    // IMAD + IMAD.HI.U32 - 6 multiplier-pipe cycles per product instead of 4; ncu round 2: 3 % of the G1 kernel's
    // executed instructions were IMAD.HI.)
    const uint32_t s[4] = {s0, s1, s2, s3};
#pragma unroll
    for (int t = 0; t < 4; t++) {
        uint64_t p = (uint64_t)s[t] * k;
        D[2 * t] = (uint32_t)p;
        D[2 * t + 1] = (uint32_t)(p >> 32);
    }
}

// D += (s0,s1,s2,s3) * k as one carry chain; returns the carry out of D[7].
LZ_HD uint32_t row_mad(uint32_t (&D)[8], uint32_t s0, uint32_t s1, uint32_t s2, uint32_t s3, uint32_t k) {
    uint32_t cy;
#ifdef __CUDA_ARCH__
    asm("mad.lo.cc.u32 %0, %9, %13, %0;\n\t"
        "madc.hi.cc.u32 %1, %9, %13, %1;\n\t"
        "madc.lo.cc.u32 %2, %10, %13, %2;\n\t"
        "madc.hi.cc.u32 %3, %10, %13, %3;\n\t"
        "madc.lo.cc.u32 %4, %11, %13, %4;\n\t"
        "madc.hi.cc.u32 %5, %11, %13, %5;\n\t"
        "madc.lo.cc.u32 %6, %12, %13, %6;\n\t"
        "madc.hi.cc.u32 %7, %12, %13, %7;\n\t"
        "addc.u32 %8, 0, 0;"
        : "+r"(D[0]), "+r"(D[1]), "+r"(D[2]), "+r"(D[3]), "+r"(D[4]), "+r"(D[5]), "+r"(D[6]), "+r"(D[7]), "=r"(cy)
        : "r"(s0), "r"(s1), "r"(s2), "r"(s3), "r"(k));
#else
    const uint32_t s[4] = {s0, s1, s2, s3};
    uint64_t c = 0;
    for (int t = 0; t < 4; t++) {
        uint64_t p = (uint64_t)s[t] * k;
        uint64_t lo = (uint64_t)D[2 * t] + (uint32_t)p + c;
        D[2 * t] = (uint32_t)lo;
        uint64_t hi = (uint64_t)D[2 * t + 1] + (uint32_t)(p >> 32) + (lo >> 32);
        D[2 * t + 1] = (uint32_t)hi;
        c = hi >> 32;
    }
    cy = (uint32_t)c;
#endif
    return cy;
}

// The per-iteration column shift of CIOS, fused with the next offset row:
//   X0 += D[1]                     (limb that drops to column 0 joins the aligned array)
//   D[j] = s*k + D[j+2] + carry    (D moves down two limbs and becomes the offset array)
// D[6..7] receive the last product plus carry only.
LZ_HD void row_mad_shift(uint32_t &X0, uint32_t (&D)[8], uint32_t s0, uint32_t s1, uint32_t s2, uint32_t s3,
                         uint32_t k) {
#ifdef __CUDA_ARCH__
    asm("add.cc.u32 %0, %0, %2;\n\t"
        "madc.lo.cc.u32 %1, %9, %13, %3;\n\t"
        "madc.hi.cc.u32 %2, %9, %13, %4;\n\t"
        "madc.lo.cc.u32 %3, %10, %13, %5;\n\t"
        "madc.hi.cc.u32 %4, %10, %13, %6;\n\t"
        "madc.lo.cc.u32 %5, %11, %13, %7;\n\t"
        "madc.hi.cc.u32 %6, %11, %13, %8;\n\t"
        "madc.lo.cc.u32 %7, %12, %13, 0;\n\t"
        "madc.hi.u32 %8, %12, %13, 0;"
        : "+r"(X0), "+r"(D[0]), "+r"(D[1]), "+r"(D[2]), "+r"(D[3]), "+r"(D[4]), "+r"(D[5]), "+r"(D[6]), "+r"(D[7])
        : "r"(s0), "r"(s1), "r"(s2), "r"(s3), "r"(k));
#else
    const uint32_t s[4] = {s0, s1, s2, s3};
    uint64_t c = (uint64_t)X0 + D[1];
    X0 = (uint32_t)c;
    c >>= 32;
    for (int t = 0; t < 4; t++) {
        uint64_t p = (uint64_t)s[t] * k;
        uint32_t alo = t < 3 ? D[2 * t + 2] : 0, ahi = t < 3 ? D[2 * t + 3] : 0;
        uint64_t lo = (uint64_t)alo + (uint32_t)p + c;
        uint64_t hi = (uint64_t)ahi + (uint32_t)(p >> 32) + (lo >> 32);
        D[2 * t] = (uint32_t)lo;
        D[2 * t + 1] = (uint32_t)hi;
        c = hi >> 32;
    }
#endif
}

// r = a + b, returns carry.  r = a - b, returns borrow (1 if a < b).
LZ_HD uint32_t add8(uint32_t (&r)[8], const uint32_t (&a)[8], const uint32_t (&b)[8]) {
    uint32_t cy;
#ifdef __CUDA_ARCH__
    asm("add.cc.u32 %0, %9, %17;\n\t"
        "addc.cc.u32 %1, %10, %18;\n\t"
        "addc.cc.u32 %2, %11, %19;\n\t"
        "addc.cc.u32 %3, %12, %20;\n\t"
        "addc.cc.u32 %4, %13, %21;\n\t"
        "addc.cc.u32 %5, %14, %22;\n\t"
        "addc.cc.u32 %6, %15, %23;\n\t"
        "addc.cc.u32 %7, %16, %24;\n\t"
        "addc.u32 %8, 0, 0;"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(cy)
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(a[4]), "r"(a[5]), "r"(a[6]), "r"(a[7]),
          "r"(b[0]), "r"(b[1]), "r"(b[2]), "r"(b[3]), "r"(b[4]), "r"(b[5]), "r"(b[6]), "r"(b[7]));
#else
    uint64_t c = 0;
    for (int i = 0; i < 8; i++) {
        c += (uint64_t)a[i] + b[i];
        r[i] = (uint32_t)c;
        c >>= 32;
    }
    cy = (uint32_t)c;
#endif
    return cy;
}

LZ_HD uint32_t sub8(uint32_t (&r)[8], const uint32_t (&a)[8], const uint32_t (&b)[8]) {
    uint32_t bw;
#ifdef __CUDA_ARCH__
    asm("sub.cc.u32 %0, %9, %17;\n\t"
        "subc.cc.u32 %1, %10, %18;\n\t"
        "subc.cc.u32 %2, %11, %19;\n\t"
        "subc.cc.u32 %3, %12, %20;\n\t"
        "subc.cc.u32 %4, %13, %21;\n\t"
        "subc.cc.u32 %5, %14, %22;\n\t"
        "subc.cc.u32 %6, %15, %23;\n\t"
        "subc.cc.u32 %7, %16, %24;\n\t"
        "subc.u32 %8, 0, 0;"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(bw)
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(a[4]), "r"(a[5]), "r"(a[6]), "r"(a[7]),
          "r"(b[0]), "r"(b[1]), "r"(b[2]), "r"(b[3]), "r"(b[4]), "r"(b[5]), "r"(b[6]), "r"(b[7]));
    bw &= 1u;   // subc of 0-0-borrow yields 0xffffffff on borrow
#else
    uint64_t c = 0;
    for (int i = 0; i < 8; i++) {
        uint64_t d = (uint64_t)a[i] - b[i] - c;
        r[i] = (uint32_t)d;
        c = (d >> 32) & 1;
    }
    bw = (uint32_t)c;
#endif
    return bw;
}

// Column accumulator (t0, t1, t2) += a * b: the 64-bit product joins (t0, t1) and the carry out joins t2.  ptxas emits
// IMAD.WIDE.U32 with a carry-OUT predicate and folds the carries of two consecutive products into one IADD3.X.
// (Measured on B200, tools/microbench/imadrate.cu: every 32x32->64 multiply-add form - plain, carry-out, carry-in
// .X, IMAD.HI - issues at the same ~31.7 lanes per SM per clock, so product and column scanning cost the same per
// limb product; column scanning is used where it needs FEWER limb products: squaring.)
LZ_HD void mac3(uint32_t &t0, uint32_t &t1, uint32_t &t2, uint32_t a, uint32_t b) {
#ifdef __CUDA_ARCH__
    asm("mad.lo.cc.u32 %0, %3, %4, %0;\n\t"
        "madc.hi.cc.u32 %1, %3, %4, %1;\n\t"
        "addc.u32 %2, %2, 0;" : "+r"(t0), "+r"(t1), "+r"(t2) : "r"(a), "r"(b));
#else
    uint64_t p = (uint64_t)a * b;
    uint64_t lo = (uint64_t)t0 + (uint32_t)p;
    uint64_t hi = (uint64_t)t1 + (uint32_t)(p >> 32) + (lo >> 32);
    t0 = (uint32_t)lo;
    t1 = (uint32_t)hi;
    t2 += (uint32_t)(hi >> 32);
#endif
}

// --------------------------------------------------------------------------
// Double-width arithmetic (lazy reduction in Fq2): a 16-limb product without reduction, and the Montgomery reduction
// of a 16-limb value, so that c0 = a0 b0 - a1 b1 and c1 = (a0+a1)(b0+b1) - a0 b0 - a1 b1 take three multiplications
// and TWO reductions (336 multiply-adds) instead of three full Montgomery products (408).
// --------------------------------------------------------------------------
// A[W..W+7] += (s0,s1,s2,s3) * k as one carry chain (pair t lands on A[W+2t], A[W+2t+1]); returns the carry out.
template <int W>
LZ_HD uint32_t row_mad_at(uint32_t (&A)[16], uint32_t s0, uint32_t s1, uint32_t s2, uint32_t s3, uint32_t k) {
    uint32_t cy;
#ifdef __CUDA_ARCH__
    asm("mad.lo.cc.u32 %0, %9, %13, %0;\n\t"
        "madc.hi.cc.u32 %1, %9, %13, %1;\n\t"
        "madc.lo.cc.u32 %2, %10, %13, %2;\n\t"
        "madc.hi.cc.u32 %3, %10, %13, %3;\n\t"
        "madc.lo.cc.u32 %4, %11, %13, %4;\n\t"
        "madc.hi.cc.u32 %5, %11, %13, %5;\n\t"
        "madc.lo.cc.u32 %6, %12, %13, %6;\n\t"
        "madc.hi.cc.u32 %7, %12, %13, %7;\n\t"
        "addc.u32 %8, 0, 0;"
        : "+r"(A[W + 0]), "+r"(A[W + 1]), "+r"(A[W + 2]), "+r"(A[W + 3]), "+r"(A[W + 4]), "+r"(A[W + 5]), "+r"(A[W + 6]),
          "+r"(A[W + 7]), "=r"(cy)
        : "r"(s0), "r"(s1), "r"(s2), "r"(s3), "r"(k));
#else
    const uint32_t s[4] = {s0, s1, s2, s3};
    uint64_t c = 0;
    for (int t = 0; t < 4; t++) {
        uint64_t pr = (uint64_t)s[t] * k;
        uint64_t lo = (uint64_t)A[W + 2 * t] + (uint32_t)pr + c;
        A[W + 2 * t] = (uint32_t)lo;
        uint64_t hi = (uint64_t)A[W + 2 * t + 1] + (uint32_t)(pr >> 32) + (lo >> 32);
        A[W + 2 * t + 1] = (uint32_t)hi;
        c = hi >> 32;
    }
    cy = (uint32_t)c;
#endif
    return cy;
}
// One b-limb of the wide product: products a_j * b_i sit at limb position i + j.  E holds the pairs that start on
// even positions, O those that start on odd positions (O[k] is position k + 1).  Windows advance by two limbs every
// two rows, so the carry out of a row always lands on a limb nothing has written yet.
template <int I>
LZ_HD void wide_row(uint32_t (&E)[16], uint32_t (&O)[16], const uint32_t (&a)[8], uint32_t k) {
    if (I % 2 == 0) {
        uint32_t ce = row_mad_at<I>(E, a[0], a[2], a[4], a[6], k);
        uint32_t co = row_mad_at<I>(O, a[1], a[3], a[5], a[7], k);
        if (I + 8 < 16) { E[I + 8] = ce; O[I + 8] = co; }
    } else {
        uint32_t co = row_mad_at<I - 1>(O, a[0], a[2], a[4], a[6], k);
        uint32_t ce = row_mad_at<I + 1>(E, a[1], a[3], a[5], a[7], k);
        if (I + 7 < 16) O[I + 7] = co;
        if (I + 9 < 16) E[I + 9] = ce;
    }
}
// T = a * b (16 limbs), a, b < 2^256
LZ_HD void mul_wide(uint32_t (&T)[16], const uint32_t (&a)[8], const uint32_t (&b)[8]) {
    uint32_t E[16], O[16];
#pragma unroll
    for (int i = 0; i < 16; i++) { E[i] = 0; O[i] = 0; }
    wide_row<0>(E, O, a, b[0]); wide_row<1>(E, O, a, b[1]); wide_row<2>(E, O, a, b[2]); wide_row<3>(E, O, a, b[3]);
    wide_row<4>(E, O, a, b[4]); wide_row<5>(E, O, a, b[5]); wide_row<6>(E, O, a, b[6]); wide_row<7>(E, O, a, b[7]);
    // T = E + (O << 32)
    T[0] = E[0];
#ifdef __CUDA_ARCH__
    asm("add.cc.u32 %0, %15, %30;\n\t"
        "addc.cc.u32 %1, %16, %31;\n\t"
        "addc.cc.u32 %2, %17, %32;\n\t"
        "addc.cc.u32 %3, %18, %33;\n\t"
        "addc.cc.u32 %4, %19, %34;\n\t"
        "addc.cc.u32 %5, %20, %35;\n\t"
        "addc.cc.u32 %6, %21, %36;\n\t"
        "addc.cc.u32 %7, %22, %37;\n\t"
        "addc.cc.u32 %8, %23, %38;\n\t"
        "addc.cc.u32 %9, %24, %39;\n\t"
        "addc.cc.u32 %10, %25, %40;\n\t"
        "addc.cc.u32 %11, %26, %41;\n\t"
        "addc.cc.u32 %12, %27, %42;\n\t"
        "addc.cc.u32 %13, %28, %43;\n\t"
        "addc.u32 %14, %29, %44;"
        : "=r"(T[1]), "=r"(T[2]), "=r"(T[3]), "=r"(T[4]), "=r"(T[5]), "=r"(T[6]), "=r"(T[7]), "=r"(T[8]), "=r"(T[9]),
          "=r"(T[10]), "=r"(T[11]), "=r"(T[12]), "=r"(T[13]), "=r"(T[14]), "=r"(T[15])
        : "r"(E[1]), "r"(E[2]), "r"(E[3]), "r"(E[4]), "r"(E[5]), "r"(E[6]), "r"(E[7]), "r"(E[8]), "r"(E[9]), "r"(E[10]),
          "r"(E[11]), "r"(E[12]), "r"(E[13]), "r"(E[14]), "r"(E[15]),
          "r"(O[0]), "r"(O[1]), "r"(O[2]), "r"(O[3]), "r"(O[4]), "r"(O[5]), "r"(O[6]), "r"(O[7]), "r"(O[8]), "r"(O[9]),
          "r"(O[10]), "r"(O[11]), "r"(O[12]), "r"(O[13]), "r"(O[14]));
#else
    uint64_t c = 0;
    for (int i = 1; i < 16; i++) {
        c += (uint64_t)E[i] + O[i - 1];
        T[i] = (uint32_t)c;
        c >>= 32;
    }
#endif
}
// r = a + b / a - b over 16 limbs; return carry / borrow
LZ_HD uint32_t add16(uint32_t (&r)[16], const uint32_t (&a)[16], const uint32_t (&b)[16]) {
    uint32_t lo_a[8], lo_b[8], hi_a[8], hi_b[8], lo[8], hi[8];
#pragma unroll
    for (int i = 0; i < 8; i++) { lo_a[i] = a[i]; lo_b[i] = b[i]; hi_a[i] = a[i + 8]; hi_b[i] = b[i + 8]; }
    uint32_t c = add8(lo, lo_a, lo_b);
    // hi = hi_a + hi_b + c
    uint32_t cv[8] = {c, 0, 0, 0, 0, 0, 0, 0}, t[8];
    uint32_t c1 = add8(t, hi_a, cv);
    uint32_t c2 = add8(hi, t, hi_b);
#pragma unroll
    for (int i = 0; i < 8; i++) { r[i] = lo[i]; r[i + 8] = hi[i]; }
    return c1 | c2;
}
LZ_HD uint32_t sub16(uint32_t (&r)[16], const uint32_t (&a)[16], const uint32_t (&b)[16]) {
    uint32_t bw;
#ifdef __CUDA_ARCH__
    asm("sub.cc.u32 %0, %17, %33;\n\t"
        "subc.cc.u32 %1, %18, %34;\n\t"
        "subc.cc.u32 %2, %19, %35;\n\t"
        "subc.cc.u32 %3, %20, %36;\n\t"
        "subc.cc.u32 %4, %21, %37;\n\t"
        "subc.cc.u32 %5, %22, %38;\n\t"
        "subc.cc.u32 %6, %23, %39;\n\t"
        "subc.cc.u32 %7, %24, %40;\n\t"
        "subc.cc.u32 %8, %25, %41;\n\t"
        "subc.cc.u32 %9, %26, %42;\n\t"
        "subc.cc.u32 %10, %27, %43;\n\t"
        "subc.cc.u32 %11, %28, %44;\n\t"
        "subc.cc.u32 %12, %29, %45;\n\t"
        "subc.cc.u32 %13, %30, %46;\n\t"
        "subc.cc.u32 %14, %31, %47;\n\t"
        "subc.cc.u32 %15, %32, %48;\n\t"
        "subc.u32 %16, 0, 0;"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(bw)
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(a[4]), "r"(a[5]), "r"(a[6]), "r"(a[7]), "r"(a[8]), "r"(a[9]),
          "r"(a[10]), "r"(a[11]), "r"(a[12]), "r"(a[13]), "r"(a[14]), "r"(a[15]),
          "r"(b[0]), "r"(b[1]), "r"(b[2]), "r"(b[3]), "r"(b[4]), "r"(b[5]), "r"(b[6]), "r"(b[7]), "r"(b[8]), "r"(b[9]),
          "r"(b[10]), "r"(b[11]), "r"(b[12]), "r"(b[13]), "r"(b[14]), "r"(b[15]));
    bw &= 1u;
#else
    uint64_t c = 0;
    for (int i = 0; i < 16; i++) {
        uint64_t d = (uint64_t)a[i] - b[i] - c;
        r[i] = (uint32_t)d;
        c = (d >> 32) & 1;
    }
    bw = (uint32_t)c;
#endif
    return bw;
}

// ---- Karatsuba for the 256 x 256 -> 512-bit product: three 128 x 128-bit products instead of four, i.e. 48 limb
// products instead of 64, paid for with ~70 add / xor instructions on the ALU pipe (which the product kernels leave
// two thirds idle: ncu round 2, sm__inst_executed_pipe_alu 36 % against a multiplier pipe at > 80 %).
//   a b = L + (L + H -+ M) B^4 + H B^8,   L = a0 b0,  H = a1 b1,  M = |a1 - a0| |b1 - b0|  (subtractive form: the middle
//   term a0 b1 + a1 b0 = L + H - (a1 - a0)(b1 - b0) needs no 129-bit operands; M is subtracted when the two
//   differences have the same sign and added otherwise).
// T[0..7] = x[0..3] * y[0..3] by column scanning (16 limb products)
LZ_HD void mul4x4(uint32_t (&T)[8], const uint32_t *x, const uint32_t *y) {
    uint32_t t0 = 0, t1 = 0, t2 = 0;
#pragma unroll
    for (int k = 0; k < 7; k++) {
#pragma unroll
        for (int i = 0; i < 4; i++) {
            const int j = k - i;
            if (j >= 0 && j < 4) mac3(t0, t1, t2, x[i], y[j]);
        }
        T[k] = t0; t0 = t1; t1 = t2; t2 = 0;
    }
    T[7] = t0;
}
// d = |x - y| over four limbs; returns an all-ones mask when x < y, else 0
LZ_HD uint32_t absdiff4(uint32_t (&d)[4], const uint32_t *x, const uint32_t *y) {
    uint32_t m;
#ifdef __CUDA_ARCH__
    asm("sub.cc.u32 %0, %5, %9;\n\t"
        "subc.cc.u32 %1, %6, %10;\n\t"
        "subc.cc.u32 %2, %7, %11;\n\t"
        "subc.cc.u32 %3, %8, %12;\n\t"
        "subc.u32 %4, 0, 0;\n\t"                 // 0 or 0xffffffff
        "xor.b32 %0, %0, %4;\n\t"
        "xor.b32 %1, %1, %4;\n\t"
        "xor.b32 %2, %2, %4;\n\t"
        "xor.b32 %3, %3, %4;\n\t"
        "sub.cc.u32 %0, %0, %4;\n\t"             // (d ^ m) - m: two's complement negation when m is all ones
        "subc.cc.u32 %1, %1, %4;\n\t"
        "subc.cc.u32 %2, %2, %4;\n\t"
        "subc.u32 %3, %3, %4;"
        : "=&r"(d[0]), "=&r"(d[1]), "=&r"(d[2]), "=&r"(d[3]), "=&r"(m)
        : "r"(x[0]), "r"(x[1]), "r"(x[2]), "r"(x[3]), "r"(y[0]), "r"(y[1]), "r"(y[2]), "r"(y[3]));
#else
    uint64_t c = 0;
    for (int i = 0; i < 4; i++) {
        uint64_t v = (uint64_t)x[i] - y[i] - c;
        d[i] = (uint32_t)v;
        c = (v >> 32) & 1;
    }
    m = c ? 0xffffffffu : 0u;
    uint64_t cy = c;
    for (int i = 0; i < 4; i++) {
        uint64_t v = (uint64_t)(d[i] ^ m) + cy;
        d[i] = (uint32_t)v;
        cy = v >> 32;
    }
#endif
    return m;
}
// T = a * b (16 limbs), a, b < 2^256
LZ_HD void mul_wide_k(uint32_t (&T)[16], const uint32_t (&a)[8], const uint32_t (&b)[8]) {
    uint32_t L[8], H[8], M[8], da[4], db[4], m8[8], mid[9];
    mul4x4(L, a, b);
    mul4x4(H, a + 4, b + 4);
    const uint32_t sa = absdiff4(da, a + 4, a), sb = absdiff4(db, b + 4, b);
    mul4x4(M, da, db);
    const uint32_t n = ~(sa ^ sb);                 // all ones: subtract M (same signs); 0: add M
    const uint32_t c = add8(m8, L, H);             // mid = L + H, 9 limbs (the ninth is the carry)
#pragma unroll
    for (int i = 0; i < 8; i++) mid[i] = m8[i];
#ifdef __CUDA_ARCH__
    // mid += (M ^ n) + (n & 1), with M ^ n sign-extended by n: mid -+ M in two's complement
    uint32_t x[8], junk;
#pragma unroll
    for (int i = 0; i < 8; i++) x[i] = M[i] ^ n;
    asm("add.cc.u32 %9, %19, 0xffffffff;\n\t"     // carry out = n & 1
        "addc.cc.u32 %0, %0, %10;\n\t"
        "addc.cc.u32 %1, %1, %11;\n\t"
        "addc.cc.u32 %2, %2, %12;\n\t"
        "addc.cc.u32 %3, %3, %13;\n\t"
        "addc.cc.u32 %4, %4, %14;\n\t"
        "addc.cc.u32 %5, %5, %15;\n\t"
        "addc.cc.u32 %6, %6, %16;\n\t"
        "addc.cc.u32 %7, %7, %17;\n\t"
        "addc.u32 %8, %18, %20;"
        : "+r"(mid[0]), "+r"(mid[1]), "+r"(mid[2]), "+r"(mid[3]), "+r"(mid[4]), "+r"(mid[5]), "+r"(mid[6]), "+r"(mid[7]),
          "=r"(mid[8]), "=&r"(junk)
        : "r"(x[0]), "r"(x[1]), "r"(x[2]), "r"(x[3]), "r"(x[4]), "r"(x[5]), "r"(x[6]), "r"(x[7]), "r"(c), "r"(n & 1u), "r"(n));
    // T = L | H, then T[4..12] += mid with the carry running to the top
    asm("add.cc.u32 %0, %12, %24;\n\t"
        "addc.cc.u32 %1, %13, %25;\n\t"
        "addc.cc.u32 %2, %14, %26;\n\t"
        "addc.cc.u32 %3, %15, %27;\n\t"
        "addc.cc.u32 %4, %16, %28;\n\t"
        "addc.cc.u32 %5, %17, %29;\n\t"
        "addc.cc.u32 %6, %18, %30;\n\t"
        "addc.cc.u32 %7, %19, %31;\n\t"
        "addc.cc.u32 %8, %20, %32;\n\t"
        "addc.cc.u32 %9, %21, 0;\n\t"
        "addc.cc.u32 %10, %22, 0;\n\t"
        "addc.u32 %11, %23, 0;"
        : "=r"(T[4]), "=r"(T[5]), "=r"(T[6]), "=r"(T[7]), "=r"(T[8]), "=r"(T[9]), "=r"(T[10]), "=r"(T[11]), "=r"(T[12]),
          "=r"(T[13]), "=r"(T[14]), "=r"(T[15])
        : "r"(L[4]), "r"(L[5]), "r"(L[6]), "r"(L[7]), "r"(H[0]), "r"(H[1]), "r"(H[2]), "r"(H[3]), "r"(H[4]), "r"(H[5]),
          "r"(H[6]), "r"(H[7]),
          "r"(mid[0]), "r"(mid[1]), "r"(mid[2]), "r"(mid[3]), "r"(mid[4]), "r"(mid[5]), "r"(mid[6]), "r"(mid[7]), "r"(mid[8]));
#pragma unroll
    for (int i = 0; i < 4; i++) T[i] = L[i];
#else
    {
        uint64_t cy = n & 1u;
        for (int i = 0; i < 8; i++) {
            cy += (uint64_t)mid[i] + (M[i] ^ n);
            mid[i] = (uint32_t)cy;
            cy >>= 32;
        }
        mid[8] = (uint32_t)(c + n + cy);
        for (int i = 0; i < 4; i++) T[i] = L[i];
        cy = 0;
        for (int i = 4; i < 16; i++) {
            const uint32_t base = i < 8 ? L[i] : H[i - 8];
            cy += (uint64_t)base + (i - 4 < 9 ? mid[i - 4] : 0u);
            T[i] = (uint32_t)cy;
            cy >>= 32;
        }
    }
#endif
}

// One round of reduce_wide, fused the way row_mad_shift fuses a product row: the limb that drops to column 0 joins
// the aligned array (A0 += D[1]), the Montgomery factor m = A0 * inv follows from it, and D moves down two limbs while
// taking the row (p1, p3, p5, p7) * m:  D[j] = p*m + D[j+2] + carry.  mul.lo leaves the carry flag alone.
LZ_HD uint32_t red_shift_row(uint32_t &A0, uint32_t (&D)[8], uint32_t p1, uint32_t p3, uint32_t p5, uint32_t p7,
                             uint32_t inv) {
    uint32_t m;
#ifdef __CUDA_ARCH__
    asm("add.cc.u32 %0, %0, %2;\n\t"
        "mul.lo.u32 %9, %0, %14;\n\t"
        "madc.lo.cc.u32 %1, %10, %9, %3;\n\t"
        "madc.hi.cc.u32 %2, %10, %9, %4;\n\t"
        "madc.lo.cc.u32 %3, %11, %9, %5;\n\t"
        "madc.hi.cc.u32 %4, %11, %9, %6;\n\t"
        "madc.lo.cc.u32 %5, %12, %9, %7;\n\t"
        "madc.hi.cc.u32 %6, %12, %9, %8;\n\t"
        "madc.lo.cc.u32 %7, %13, %9, 0;\n\t"
        "madc.hi.u32 %8, %13, %9, 0;"
        : "+r"(A0), "+r"(D[0]), "+r"(D[1]), "+r"(D[2]), "+r"(D[3]), "+r"(D[4]), "+r"(D[5]), "+r"(D[6]), "+r"(D[7]), "=&r"(m)
        : "r"(p1), "r"(p3), "r"(p5), "r"(p7), "r"(inv));
#else
    const uint32_t s[4] = {p1, p3, p5, p7};
    uint64_t c = (uint64_t)A0 + D[1];
    A0 = (uint32_t)c;
    c >>= 32;
    m = A0 * inv;
    for (int t = 0; t < 4; t++) {
        uint64_t pr = (uint64_t)s[t] * m;
        uint32_t alo = t < 3 ? D[2 * t + 2] : 0, ahi = t < 3 ? D[2 * t + 3] : 0;
        uint64_t lo = (uint64_t)alo + (uint32_t)pr + c;
        uint64_t hi = (uint64_t)ahi + (uint32_t)(pr >> 32) + (lo >> 32);
        D[2 * t] = (uint32_t)lo;
        D[2 * t + 1] = (uint32_t)hi;
        c = hi >> 32;
    }
#endif
    return m;
}

// T += p * 2^256 if neg (T is a difference of products that came out negative, above -p * 2^256)
template <class P>
LZ_HD void wide_fix_negative(uint32_t (&T)[16], uint32_t neg) {
    uint32_t hi[8], pm[8], fix[8];
#pragma unroll
    for (int i = 0; i < 8; i++) { hi[i] = T[8 + i]; pm[i] = neg ? P::MOD(i) : 0u; }
    add8(fix, hi, pm);
#pragma unroll
    for (int i = 0; i < 8; i++) T[8 + i] = fix[i];
}

// --------------------------------------------------------------------------
// Field element.  P supplies INV, MOD(i), ONE(i), R2(i), ...
// --------------------------------------------------------------------------
template <class P>
struct alignas(16) Fp {
    uint32_t l[8];

    LZ_HD static Fp zero() {
        Fp r;
#pragma unroll
        for (int i = 0; i < 8; i++) r.l[i] = 0;
        return r;
    }
    LZ_HD static Fp one() {
        Fp r;
#pragma unroll
        for (int i = 0; i < 8; i++) r.l[i] = P::ONE(i);
        return r;
    }
    LZ_HD static Fp modulus() {
        Fp r;
#pragma unroll
        for (int i = 0; i < 8; i++) r.l[i] = P::MOD(i);
        return r;
    }
    LZ_HD static Fp r2() {
        Fp r;
#pragma unroll
        for (int i = 0; i < 8; i++) r.l[i] = P::R2(i);
        return r;
    }
    LZ_HD bool is_zero() const {
        uint32_t o = 0;
#pragma unroll
        for (int i = 0; i < 8; i++) o |= l[i];
        return o == 0;
    }
    LZ_HD bool operator==(const Fp &b) const {
        uint32_t o = 0;
#pragma unroll
        for (int i = 0; i < 8; i++) o |= l[i] ^ b.l[i];
        return o == 0;
    }
    LZ_HD bool operator!=(const Fp &b) const { return !(*this == b); }

    // r = x - p if x >= p else x   (x < 2p)
    LZ_HD static Fp reduce_once(const uint32_t (&x)[8]) {
        Fp m = modulus(), d, r;
        uint32_t bw = sub8(d.l, x, m.l);
#pragma unroll
        for (int i = 0; i < 8; i++) r.l[i] = bw ? x[i] : d.l[i];
        return r;
    }
    LZ_HD friend Fp operator+(const Fp &a, const Fp &b) {
        uint32_t s[8];
        add8(s, a.l, b.l);      // p < 2^254: no carry out
        return reduce_once(s);
    }
    LZ_HD friend Fp operator-(const Fp &a, const Fp &b) {
        Fp d, e, m = modulus(), r;
        uint32_t bw = sub8(d.l, a.l, b.l);
        add8(e.l, d.l, m.l);
#pragma unroll
        for (int i = 0; i < 8; i++) r.l[i] = bw ? e.l[i] : d.l[i];
        return r;
    }
    LZ_HD Fp neg() const {
        Fp m = modulus(), d, r;
        sub8(d.l, m.l, l);
        bool z = is_zero();
#pragma unroll
        for (int i = 0; i < 8; i++) r.l[i] = z ? 0u : d.l[i];
        return r;
    }
    LZ_HD Fp dbl() const { return *this + *this; }

    // Montgomery product a*b*R^-1 mod p.
    LZ_HD friend Fp operator*(const Fp &a, const Fp &b) { return reduce_once(mul_lazy(a, b).l); }
    LZ_HD Fp sqr() const { return reduce_once(sqr_lazy().l); }
    // Montgomery reduction of a 16-limb T < p * 2^256, canonical result.
    LZ_HD static Fp reduce_wide(const uint32_t (&T)[16]) { return reduce_once(reduce_wide_lazy(T).l); }
    // a*b - c*d with ONE reduction (the Y3 of every XYZZ formula), a, b, c, d < p.  200 multiply-adds instead of 272.
    LZ_HD static Fp msub(const Fp &a, const Fp &b, const Fp &c, const Fp &d) { return reduce_once(msub_lazy(a, b, c, d).l); }

    // ---- Redundant form: values in [0, 2p) instead of [0, p), for the G1 table-gather kernel's mixed addition
    // (ec.cuh madd_lazy).  The primitives below are the cores of the canonical operations without their final
    // conditional subtraction (8 subtractions + 8 selects each).  BN254's p = 0.18903 R (R = 2^256), so 4p < R and
    // the Montgomery reduction still returns below 2p from operands below 2p: the bound of every result is stated
    // beside it.  Units below: multiples of p, with R = 5.29 p.
    //
    // CIOS product without the final subtraction: (a b + m p) / R < a b / R + p for any a < R - p (the accumulator,
    // at most (a + p) 2^32 before each shift, stays below 2^288) and any b < R.  a, b < 2p: < 1.76p; a < p, b < 2p:
    // < 1.38p; generally < 2p whenever a b < p R.
    LZ_HD static Fp mul_lazy(const Fp &a, const Fp &b) {
        uint32_t X[8], Y[8];      // aligned / offset accumulators (roles swap every iteration)
        uint32_t m, c;
        // i = 0
        row_mul(X, a.l[0], a.l[2], a.l[4], a.l[6], b.l[0]);
        row_mul(Y, a.l[1], a.l[3], a.l[5], a.l[7], b.l[0]);
        m = X[0] * P::INV;
        row_mad(Y, P::MOD(1), P::MOD(3), P::MOD(5), P::MOD(7), m);
        c = row_mad(X, P::MOD(0), P::MOD(2), P::MOD(4), P::MOD(6), m);
        Y[7] += c;
#pragma unroll
        for (int i = 1; i < 8; i++) {
            if (i & 1) {
                // X was just reduced (X[0] == 0): Y becomes aligned, X shifts into the offset role.
                row_mad_shift(Y[0], X, a.l[1], a.l[3], a.l[5], a.l[7], b.l[i]);
                c = row_mad(Y, a.l[0], a.l[2], a.l[4], a.l[6], b.l[i]);
                X[7] += c;
                m = Y[0] * P::INV;
                row_mad(X, P::MOD(1), P::MOD(3), P::MOD(5), P::MOD(7), m);
                c = row_mad(Y, P::MOD(0), P::MOD(2), P::MOD(4), P::MOD(6), m);
                X[7] += c;
            } else {
                row_mad_shift(X[0], Y, a.l[1], a.l[3], a.l[5], a.l[7], b.l[i]);
                c = row_mad(X, a.l[0], a.l[2], a.l[4], a.l[6], b.l[i]);
                Y[7] += c;
                m = X[0] * P::INV;
                row_mad(Y, P::MOD(1), P::MOD(3), P::MOD(5), P::MOD(7), m);
                c = row_mad(X, P::MOD(0), P::MOD(2), P::MOD(4), P::MOD(6), m);
                Y[7] += c;
            }
        }
        // After i = 7 (odd): Y aligned with Y[0] == 0, X offset.  result = X + (Y >> 32).
        uint32_t hi[8];
#pragma unroll
        for (int j = 0; j < 7; j++) hi[j] = Y[j + 1];
        hi[7] = 0;
        Fp s;
        add8(s.l, X, hi);
        return s;
    }
    // a^2 * R^-1 by column scanning with the reduction interleaved (FIPS): 36 + 64 limb products instead of 64 + 64.
    //   a^2 = sum_i a_i B^i * (a_i B^i + 2 * (a div B^(i+1)) * B^(i+1)):  row i multiplies a_i by a_i, by
    //   e_(i+1) = 2 a_(i+1) mod 2^32 (bit 0 clear) and by d_j = limb j of 2a (j > i + 1); 2a < 2^256 because a < 2^255.
    // Measured 79 G squarings/s against 64 G products/s (tools/microbench/mulcs.cu), bit-exact against operator*.
    // Without the final subtraction: a < 2^255 (= 2.64p), result < a^2 / R + p; a < 2p: < 1.76p.
    LZ_HD Fp sqr_lazy() const {
#ifdef LZKP_SQR_AS_MUL           // A/B switch: the round-1 behaviour (a full product)
        return mul_lazy(*this, *this);
#endif
        uint32_t d[8], e[8];
        d[0] = l[0] << 1;
        e[0] = 0;
#pragma unroll
        for (int i = 1; i < 8; i++) { d[i] = (l[i] << 1) | (l[i - 1] >> 31); e[i] = l[i] << 1; }
        uint32_t t0 = 0, t1 = 0, t2 = 0, m[8];
        Fp r;
#pragma unroll
        for (int k = 0; k < 15; k++) {
#pragma unroll
            for (int i = 0; i < 8; i++) {
                const int j = k - i;
                if (j < i || j > 7) continue;
                if (j == i) mac3(t0, t1, t2, l[i], l[i]);
                else if (j == i + 1) mac3(t0, t1, t2, l[i], e[j]);
                else mac3(t0, t1, t2, l[i], d[j]);
            }
            if (k < 8) {
#pragma unroll
                for (int i = 0; i < k; i++) mac3(t0, t1, t2, m[i], P::MOD(k - i));
                m[k] = t0 * P::INV;
                mac3(t0, t1, t2, m[k], P::MOD(0));
            } else {
#pragma unroll
                for (int i = k - 7; i < 8; i++) mac3(t0, t1, t2, m[i], P::MOD(k - i));
                r.l[k - 8] = t0;
            }
            t0 = t1; t1 = t2; t2 = 0;
        }
        r.l[7] = t0;
        return r;
    }
    // Montgomery reduction of a 16-limb T < p * 2^256 without the final subtraction: T * R^-1 mod p =
    // (T_lo + M p) / R + T_hi, where the eight rounds run on the lower half alone (U = (T_lo + M p) / R <= p) in the
    // product's aligned / offset accumulators, and T_hi < p joins at the end: U + T_hi < 2p.
    LZ_HD static Fp reduce_wide_lazy(const uint32_t (&T)[16]) {
        uint32_t X[8], Y[8];
        uint32_t m, c;
#pragma unroll
        for (int j = 0; j < 8; j++) X[j] = T[j];
        m = X[0] * P::INV;
        row_mul(Y, P::MOD(1), P::MOD(3), P::MOD(5), P::MOD(7), m);
        c = row_mad(X, P::MOD(0), P::MOD(2), P::MOD(4), P::MOD(6), m);
        Y[7] += c;
#pragma unroll
        for (int i = 1; i < 8; i++) {
            if (i & 1) {
                m = red_shift_row(Y[0], X, P::MOD(1), P::MOD(3), P::MOD(5), P::MOD(7), P::INV);
                c = row_mad(Y, P::MOD(0), P::MOD(2), P::MOD(4), P::MOD(6), m);
                X[7] += c;
            } else {
                m = red_shift_row(X[0], Y, P::MOD(1), P::MOD(3), P::MOD(5), P::MOD(7), P::INV);
                c = row_mad(X, P::MOD(0), P::MOD(2), P::MOD(4), P::MOD(6), m);
                Y[7] += c;
            }
        }
        // after i = 7: Y aligned with Y[0] == 0, X offset: U = X + (Y >> 32)
        uint32_t hi[8], th[8], u[8];
#pragma unroll
        for (int j = 0; j < 7; j++) hi[j] = Y[j + 1];
        hi[7] = 0;
#pragma unroll
        for (int j = 0; j < 8; j++) th[j] = T[8 + j];
        add8(u, X, hi);
        Fp s_;
        add8(s_.l, u, th);
        return s_;
    }
    // a*b - c*d as two 16-limb products, the difference brought back into [0, p * 2^256) by adding p * 2^256 when
    // negative, and one reduction without the final subtraction.  a b < p R and c d < p R (all four below 2p: 4p^2 =
    // 0.76 p R): result < 2p.
    LZ_HD static Fp msub_lazy(const Fp &a, const Fp &b, const Fp &c, const Fp &d) {
        uint32_t t0[16], t1[16];
        mul_wide(t0, a.l, b.l);
        mul_wide(t1, c.l, d.l);
        const uint32_t bw = sub16(t0, t0, t1);
        wide_fix_negative<P>(t0, bw);
        return reduce_wide_lazy(t0);
    }
    // a - b, plus 2p when negative:  a, b < 2p -> [0, 2p)
    LZ_HD static Fp sub_2p(const Fp &a, const Fp &b) {
        Fp d, e, r;
        uint32_t bw = sub8(d.l, a.l, b.l);
        add8(e.l, d.l, modulus2().l);
#pragma unroll
        for (int i = 0; i < 8; i++) r.l[i] = bw ? e.l[i] : d.l[i];
        return r;
    }
    // a + b, less 2p when at least 2p:  a, b < 2p -> [0, 2p)
    LZ_HD static Fp add_2p(const Fp &a, const Fp &b) {
        uint32_t s[8];
        Fp d, r;
        add8(s, a.l, b.l);        // a + b < 4p < 2^256: no carry out
        uint32_t bw = sub8(d.l, s, modulus2().l);
#pragma unroll
        for (int i = 0; i < 8; i++) r.l[i] = bw ? s[i] : d.l[i];
        return r;
    }
    // x == 0 mod p for x < 2p: x is 0 or p
    LZ_HD bool is_zero_2p() const {
        uint32_t z = 0, q = 0;
#pragma unroll
        for (int i = 0; i < 8; i++) { z |= l[i]; q |= l[i] ^ P::MOD(i); }
        return z == 0 || q == 0;
    }
    // [0, 2p) -> [0, p)
    LZ_HD Fp canonical() const { return reduce_once(l); }
    LZ_HD static Fp modulus2() {
        Fp r;
#pragma unroll
        for (int i = 0; i < 8; i++) r.l[i] = (P::MOD(i) << 1) | (i ? P::MOD(i - 1) >> 31 : 0u);
        return r;
    }

    // canonical (plain integer, < p) <-> Montgomery
    LZ_HD static Fp from_canonical(const Fp &c) { return c * r2(); }
    LZ_HD Fp to_canonical() const {
        Fp o = zero();
        o.l[0] = 1;
        return *this * o;
    }
    // Inverse by the binary extended Euclidean algorithm (HAC 14.61 for an odd modulus); 0 -> 0.
    // ~750 shift / add / subtract steps on 256-bit integers: about 5x shorter as a serial chain than the
    // Fermat ladder (254 squarings + 127 products), which matters because every use is latency-bound
    // (3 per proof in k_assemble, 1 per MSM result, 1 per table entry group).  Works on the limbs as a
    // plain integer, so for a Montgomery input aR it yields (aR)^-1; one product with R^3 restores a^-1 R.
    LZ_COLD Fp inverse() const {
        if (is_zero()) return zero();
        uint32_t u[8], v[8], x1[8], x2[8];
        const Fp m = modulus();
#pragma unroll
        for (int i = 0; i < 8; i++) { u[i] = l[i]; v[i] = m.l[i]; x1[i] = 0; x2[i] = 0; }
        x1[0] = 1;
        auto is_one = [](const uint32_t (&a)[8]) {
            uint32_t o = a[0] ^ 1u;
#pragma unroll
            for (int i = 1; i < 8; i++) o |= a[i];
            return o == 0;
        };
        auto shr1 = [](uint32_t (&a)[8]) {
#pragma unroll
            for (int i = 0; i < 7; i++) a[i] = (a[i] >> 1) | (a[i + 1] << 31);
            a[7] >>= 1;
        };
        auto halve_mod = [&](uint32_t (&x)[8]) {          // x / 2 mod p, x < p
            if (x[0] & 1u) { uint32_t t[8]; add8(t, x, m.l); 
#pragma unroll
                for (int i = 0; i < 8; i++) x[i] = t[i]; }
            shr1(x);
        };
        auto sub_mod = [&](uint32_t (&x)[8], const uint32_t (&y)[8]) {   // x = x - y mod p
            uint32_t d[8], e[8];
            uint32_t bw = sub8(d, x, y);
            add8(e, d, m.l);
#pragma unroll
            for (int i = 0; i < 8; i++) x[i] = bw ? e[i] : d[i];
        };
#pragma unroll 1
        while (!is_one(u) && !is_one(v)) {
#pragma unroll 1
            while (!(u[0] & 1u)) { shr1(u); halve_mod(x1); }
#pragma unroll 1
            while (!(v[0] & 1u)) { shr1(v); halve_mod(x2); }
            uint32_t d[8];
            if (sub8(d, u, v) == 0) {                       // u >= v
#pragma unroll
                for (int i = 0; i < 8; i++) u[i] = d[i];
                sub_mod(x1, x2);
            } else {
                sub8(d, v, u);
#pragma unroll
                for (int i = 0; i < 8; i++) v[i] = d[i];
                sub_mod(x2, x1);
            }
        }
        Fp r, r3;
        const bool uu = is_one(u);
#pragma unroll
        for (int i = 0; i < 8; i++) { r.l[i] = uu ? x1[i] : x2[i]; r3.l[i] = P::R3(i); }
        return r * r3;
    }
    // canonical a > b ?
    LZ_HD static bool gt_canonical(const Fp &a, const Fp &b) {
        uint32_t d[8];
        return sub8(d, b.l, a.l) != 0;   // b - a borrows  <=>  a > b
    }
};

using Fr = Fp<FrParams>;
using Fq = Fp<FqParams>;

// --------------------------------------------------------------------------
// Fq2 = Fq[u]/(u^2 + 1)
// --------------------------------------------------------------------------
struct Fq2;
#if !defined(LZKP_FQ2_INLINE) && defined(__CUDA_ARCH__)
static __device__ __noinline__ Fq2 fq2_mul_call(Fq2 a, Fq2 b);
static __device__ __noinline__ Fq2 fq2_sqr_call(Fq2 a);
#endif
struct Fq2 {
    Fq c0, c1;
    LZ_HD static Fq2 zero() { return Fq2{Fq::zero(), Fq::zero()}; }
    LZ_HD static Fq2 one() { return Fq2{Fq::one(), Fq::zero()}; }
    LZ_HD bool is_zero() const { return c0.is_zero() && c1.is_zero(); }
    LZ_HD bool operator==(const Fq2 &b) const { return c0 == b.c0 && c1 == b.c1; }
    LZ_HD bool operator!=(const Fq2 &b) const { return !(*this == b); }
    LZ_HD friend Fq2 operator+(const Fq2 &a, const Fq2 &b) { return Fq2{a.c0 + b.c0, a.c1 + b.c1}; }
    LZ_HD friend Fq2 operator-(const Fq2 &a, const Fq2 &b) { return Fq2{a.c0 - b.c0, a.c1 - b.c1}; }
    LZ_HD Fq2 neg() const { return Fq2{c0.neg(), c1.neg()}; }
    LZ_HD Fq2 dbl() const { return Fq2{c0.dbl(), c1.dbl()}; }
    LZ_HD friend Fq2 operator*(const Fq2 &a, const Fq2 &b) {
#if !defined(LZKP_FQ2_INLINE) && defined(__CUDA_ARCH__)
        return fq2_mul_call(a, b);
#elif defined(LZKP_FQ2_SCHOOLBOOK)
        // four independent products, two additions: more multiplies than Karatsuba but no dependent add chains
        return Fq2{a.c0 * b.c0 - a.c1 * b.c1, a.c0 * b.c1 + a.c1 * b.c0};
#else
        Fq v0 = a.c0 * b.c0, v1 = a.c1 * b.c1;                 // Karatsuba, 3 Fq products
        Fq s = (a.c0 + a.c1) * (b.c0 + b.c1);
        return Fq2{v0 - v1, s - v0 - v1};
#endif
    }
    LZ_HD Fq2 sqr() const {                                     // 2 Fq products
#if !defined(LZKP_FQ2_INLINE) && defined(__CUDA_ARCH__)
        return fq2_sqr_call(*this);
#endif
        Fq m = c0 * c1;
        return Fq2{(c0 + c1) * (c0 - c1), m.dbl()};
    }
    // a*b - c*d.  (Sharing the reductions between the two products, as Fp::msub does, was measured SLOWER here: as a
    // four-operand out-of-line call it moves 64 registers of arguments, -7 % on the G2 gather kernel.)
    LZ_HD static Fq2 msub(const Fq2 &a, const Fq2 &b, const Fq2 &c, const Fq2 &d) { return a * b - c * d; }
    LZ_HD Fq2 inverse() const {
        Fq n = (c0.sqr() + c1.sqr()).inverse();
        return Fq2{c0 * n, (c1 * n).neg()};
    }
};
// Karatsuba with lazy reduction: three 16-limb products, two Montgomery reductions.
//   c1 = (a0 + a1)(b0 + b1) - a0 b0 - a1 b1 = a0 b1 + a1 b0 in [0, 2 p^2)            (the sums stay unreduced, < 2^255)
//   c0 = a0 b0 - a1 b1, plus p * 2^256 when negative,        in [0, p * 2^256)
// both below p * 2^256, so reduce_wide returns the canonical Montgomery residues.
LZ_HD Fq2 fq2_mul_lazy(const Fq2 &a, const Fq2 &b) {
    uint32_t t0[16], t1[16], t2[16], sa[8], sb[8];
    mul_wide(t0, a.c0.l, b.c0.l);
    mul_wide(t1, a.c1.l, b.c1.l);
    add8(sa, a.c0.l, a.c1.l);
    add8(sb, b.c0.l, b.c1.l);
    mul_wide(t2, sa, sb);
    sub16(t2, t2, t0);
    sub16(t2, t2, t1);
    const uint32_t bw = sub16(t0, t0, t1);
    uint32_t hi[8], pm[8], fix[8];
#pragma unroll
    for (int i = 0; i < 8; i++) { hi[i] = t0[8 + i]; pm[i] = bw ? FqParams::MOD(i) : 0u; }
    add8(fix, hi, pm);
#pragma unroll
    for (int i = 0; i < 8; i++) t0[8 + i] = fix[i];
    return Fq2{Fq::reduce_wide(t0), Fq::reduce_wide(t2)};
}
#if !defined(LZKP_FQ2_INLINE) && defined(__CUDA_ARCH__)
// Out-of-line Fq2 product / square (operands and result in registers).  A G2 mixed addition with its 28 Montgomery
// products inlined is ~110 KB of SASS, more than the instruction cache holds: ncu showed 11 % of the G2 gather
// kernel's stall samples as no_instruction.  As calls the loop body is ~15 KB; measured -19 % on the G2 bucket
// accumulation and -5 % on the G2 table-gather kernel.  -DLZKP_FQ2_INLINE restores the inlined form.
static __device__ __noinline__ Fq2 fq2_mul_call(Fq2 a, Fq2 b) { return fq2_mul_lazy(a, b); }
static __device__ __noinline__ Fq2 fq2_sqr_call(Fq2 a) {
    Fq m = a.c0 * a.c1;
    return Fq2{(a.c0 + a.c1) * (a.c0 - a.c1), m.dbl()};
}
#endif

}  // namespace lzkp
