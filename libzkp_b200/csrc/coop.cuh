// coop.cuh — warp-cooperative BN254 pairing arithmetic: the latency form of the verifier (SURVEY.md §8f-3).
//
// k_verify4 (verify.cu) runs one proof per LANE: right for throughput, but a single verification is then one
// thread's dependent chain of ~20 000 field products (13.7 ms, against ~3 ms for arkworks on a CPU, which is what the
// reference pays per call at src/backend/snark.rs:377-401).  A warp instruction costs the same whether 1 or 32 lanes
// are active, so here ONE proof owns a CTA and both the lanes of a warp and the warps share the work:
//   * f12_mul: the 18 Fq2 products of a Karatsuba Fq12 product (3 Fq6 products of 6) run on 18 lanes at once; the
//     recombination runs on 10 and then 6 lanes.  Squarings, cyclotomic squarings and line products all use this one
//     body (lines as dense operands with zero slots) - in the latency regime a cheaper formula on fewer lanes buys
//     nothing, and a second body only widens the instruction footprint of a loop a lone warp runs.
//   * the Miller loop of (A, B) runs on three warps: line_chain walks the twist point (the dependent chain of G2
//     doublings / additions, 3-4 product rounds each) and publishes scaled line coefficients in shared memory; two
//     warps fold them into f, each running a share of the loop (miller_f, kMillerSplit).  The loops against -gamma,
//     -delta (and beta, for the combined check of verify.cu) read line coefficients PREPARED at lzkp_vk_load (what
//     ark-groth16's PreparedVerifyingKey holds) and scale them on idle lanes of the previous product.
//   * vk_x = gamma_abc_0 + sum x_i gamma_abc_i comes from fixed-base byte-window tables built at lzkp_vk_load
//     (lane = (input, byte) pair, then a shuffle tree).
//   * the r-torsion test of B (one 63-bit ladder, pairing.cuh g2_subgroup_from_xp) runs with the independent products of
//     every doubling / addition on different lanes, beside the Miller loops and the final exponentiation.
//   * the final exponentiation's three powers by x are split into a squaring warp and a multiplying warp
//     (f12_exp_neg_x / f12_exp_helper).
// Warps talk through counters in shared memory polled with __nanosleep back-off (flag_publish / flag_wait).
// Same formulas as pairing.cuh (the serial code is the checker: LZKP_COOP_SELFTEST=1 compares both at key load).
#pragma once
#include "dev_util.cuh"
#include "pairing.cuh"

namespace lzkp {
namespace coop {

LZ_HD constexpr int popcnt64(uint64_t v) {
    int c = 0;
    for (int i = 0; i < 64; i++) c += (int)((v >> i) & 1ull);
    return c;
}
constexpr int kLines = (kAteTop + 1) + popcnt64(kAteNafNz) + 2;   // doublings + additions (NAF digits of 6x + 2) + the two Frobenius additions
constexpr uint32_t kTabDigits = 255, kTabWindows = 32;        // byte windows of a canonical 32-byte scalar

__device__ __forceinline__ int lane_id() { return (int)(threadIdx.x & 31u); }
__device__ __forceinline__ Fq2 ldq(const Fq2 *p) { return ld_vec(p); }
__device__ __forceinline__ void stq(Fq2 *p, const Fq2 &v) { st_vec(p, v); }
__device__ __forceinline__ Fq fq_half(const Fq &a) {          // a / 2 mod p on the residue itself (any representation)
    const Fq m = Fq::modulus();
    uint32_t mm[8], t[8];
    const bool odd = (a.l[0] & 1u) != 0;
#pragma unroll
    for (int i = 0; i < 8; i++) mm[i] = odd ? m.l[i] : 0u;
    add8(t, a.l, mm);                                         // a + p < 2^255
    Fq r;
#pragma unroll
    for (int i = 0; i < 7; i++) r.l[i] = (t[i] >> 1) | (t[i + 1] << 31);
    r.l[7] = t[7] >> 1;
    return r;
}
__device__ __forceinline__ Fq2 fq2_half(const Fq2 &a) { return Fq2{fq_half(a.c0), fq_half(a.c1)}; }
__device__ __forceinline__ Fq2 fq2_triple(const Fq2 &a) { return a.dbl() + a; }
__device__ __forceinline__ Fq2 fq2_embed(const Fq &a) { return Fq2{a, Fq::zero()}; }

// Fq2 additions of the linear phases.  (Measured: as out-of-line calls - 3x less code - a single verification takes
// 2.81 ms instead of 2.50: a lone warp is bound by its dependent instruction count, not by instruction fetch.)
#define LZ_COOP_OP __device__ __forceinline__
LZ_COOP_OP Fq2 qadd(Fq2 a, Fq2 b) { return a + b; }
LZ_COOP_OP Fq2 qsub(Fq2 a, Fq2 b) { return a - b; }
LZ_COOP_OP Fq2 qxi(Fq2 a) { return fq2_mul_xi(a); }

// An Fq12 value is six Fq2 coefficients in tower order: index 3h + k is coefficient v^k of c_h (struct Fq12's layout).
struct Scratch {
    Fq2 P[19];      // the Karatsuba products; P[18] stays zero (scratch_init)
    Fq2 T[10];      // Fq6-level sums
};

// coefficient v^k of c_h of b; SPARSE: b is a line (l0, l1, l2) = l0 + l1 w + l2 v w
template <bool SPARSE>
__device__ __forceinline__ Fq2 coeff(const Fq2 *b, int h, int k) {
    if (!SPARSE) return ldq(b + 3 * h + k);
    if (h == 0) return k == 0 ? ldq(b) : Fq2::zero();
    return k < 2 ? ldq(b + 1 + k) : Fq2::zero();
}
template <bool SPARSE>
__device__ __forceinline__ Fq2 operand(const Fq2 *b, int X, int i) {      // coefficient i of (c0, c1, c0 + c1)[X]
    Fq2 s = coeff<SPARSE>(b, X == 1 ? 1 : 0, i);
    if (X == 2) s = qadd(s, coeff<SPARSE>(b, 1, i));
    return s;
}

// r = a * b.  Every lane of the warp calls; r may alias a or b.  Lanes 18.. may carry one extra Fq2 product each
// (*so = *sa * *sb, so == nullptr: none) that rides in the same instruction stream.
#ifdef LZKP_COOP_PROF          // per-phase cycle counters of f12_mul (variant build only; warp 0 of CTA 0)
__device__ long long g_coop_prof[8];
#define LZ_PROF_T(k) const long long prof_t##k = clock64()
#define LZ_PROF_ADD(i, k0, k1) if (threadIdx.x == 0 && blockIdx.x == 0) g_coop_prof[i] += prof_t##k1 - prof_t##k0
#else
#define LZ_PROF_T(k)
#define LZ_PROF_ADD(i, k0, k1)
#endif
template <bool SPARSE>
__device__ __noinline__ void f12_mul(Fq2 *r, const Fq2 *a, const Fq2 *b, Scratch *s, const Fq2 *sa = nullptr,
                                     const Fq2 *sb = nullptr, Fq2 *so = nullptr) {
    const int lane = lane_id();
    LZ_PROF_T(0);
    Fq2 x = Fq2::zero(), y = Fq2::zero();
    const bool same = !SPARSE && a == b;             // a squaring (warp-uniform): the operand sums are computed once
    if (lane < 18) {
        const int X = lane / 6, j = lane - 6 * X;
        const int i1 = j < 3 ? j : (j == 3 ? 1 : 0), i2 = j < 3 ? -1 : (j == 4 ? 1 : 2);
        x = operand<false>(a, X, i1);
        if (!same) y = operand<SPARSE>(b, X, i1);
        if (i2 >= 0) {
            x = qadd(x, operand<false>(a, X, i2));
            if (!same) y = qadd(y, operand<SPARSE>(b, X, i2));
        }
        if (same) y = x;
    } else if (so) {
        x = ldq(sa);
        y = ldq(sb);
    }
    __syncwarp();
    LZ_PROF_T(1);
    const Fq2 p = x * y;
    __syncwarp();
    LZ_PROF_T(2);
    if (lane < 18) stq(&s->P[lane], p);
    else if (so) stq(so, p);
    __syncwarp();
    // Fq6 level, one instruction stream for all ten lanes:  w = P[i0] - P[i1] - P[i2] + P[i3];  t = base + xi * e
    //   T[3X+0] = P0 + xi (P3 - P1 - P2)      T[3X+1] = (P4 - P0 - P1) + xi P2      T[3X+2] = P5 - P0 - P2 + P1
    //   T[9]    = xi * T[5] = xi (P11 - P6 - P8 + P7)
    if (lane < 10) {
        const int X = lane == 9 ? 1 : lane / 3, k = lane == 9 ? 3 : lane - 3 * X;
        const int o = 6 * X, zi = 18;        // zi: the zero slot
        const int i0 = k == 0 ? o + 3 : k == 1 ? o + 4 : k == 2 ? o + 5 : 11;
        const int i1 = k == 0 ? o + 1 : k == 3 ? 6 : o + 0;
        const int i2 = k == 0 ? o + 2 : k == 1 ? o + 1 : k == 2 ? o + 2 : 8;
        const int i3 = k == 2 ? o + 1 : k == 3 ? 7 : zi;
        const Fq2 w = qadd(qsub(qsub(ldq(&s->P[i0]), ldq(&s->P[i1])), ldq(&s->P[i2])), ldq(&s->P[i3]));
        const Fq2 other = ldq(&s->P[k == 0 ? o + 0 : k == 1 ? o + 2 : zi]);   // k = 0: the base P0, k = 1: e = P2
        const bool e_is_w = (k == 0) | (k == 3);
        Fq2 e, base;
#pragma unroll
        for (int i = 0; i < 8; i++) {
            e.c0.l[i] = e_is_w ? w.c0.l[i] : other.c0.l[i];
            e.c1.l[i] = e_is_w ? w.c1.l[i] : other.c1.l[i];
            base.c0.l[i] = k == 0 ? other.c0.l[i] : (k == 3 ? 0u : w.c0.l[i]);
            base.c1.l[i] = k == 0 ? other.c1.l[i] : (k == 3 ? 0u : w.c1.l[i]);
        }
        stq(&s->T[lane], qadd(base, qxi(e)));      // k = 2: e = 0
    }
    __syncwarp();
    LZ_PROF_T(3);
    // Fq12 level:  c0 = T0 + v T1 = (T0[0] + xi T1[2], T0[1] + T1[0], T0[2] + T1[1]),  c1 = T2 - T0 - T1
    if (lane < 6) {
        Fq2 t;
        if (lane < 3) t = qadd(ldq(&s->T[lane]), ldq(&s->T[lane == 0 ? 9 : 2 + lane]));
        else t = qsub(qsub(ldq(&s->T[3 + lane]), ldq(&s->T[lane - 3])), ldq(&s->T[lane]));
        stq(r + lane, t);
    }
    __syncwarp();
    LZ_PROF_T(4);
    LZ_PROF_ADD(0, 0, 1); LZ_PROF_ADD(1, 1, 2); LZ_PROF_ADD(2, 2, 3); LZ_PROF_ADD(3, 3, 4);
#ifdef LZKP_COOP_PROF
    if (threadIdx.x == 0 && blockIdx.x == 0) g_coop_prof[4] += 1;
#endif
}

__device__ __forceinline__ void f12_set_one(Fq2 *f) {
    const int lane = lane_id();
    if (lane < 6) stq(f + lane, lane == 0 ? Fq2::one() : Fq2::zero());
    __syncwarp();
}
__device__ __forceinline__ void f12_copy(Fq2 *d, const Fq2 *a) {
    const int lane = lane_id();
    Fq2 v = Fq2::zero();
    if (lane < 6) v = ldq(a + lane);
    __syncwarp();
    if (lane < 6) stq(d + lane, v);
    __syncwarp();
}
__device__ __forceinline__ void f12_conj(Fq2 *d, const Fq2 *a) {
    const int lane = lane_id();
    Fq2 v = Fq2::zero();
    if (lane < 6) { v = ldq(a + lane); if (lane >= 3) v = v.neg(); }
    __syncwarp();
    if (lane < 6) stq(d + lane, v);
    __syncwarp();
}
// x -> x^(p^K), K = 1, 2, 3: one product per coefficient (K odd: of the conjugate).  Constant of index 3h + k:
// xi^((p^K - 1)(2k + h)/6).
template <int K>
__device__ __noinline__ void f12_frob(Fq2 *d, const Fq2 *a) {
    const int lane = lane_id();
    Fq2 x = Fq2::zero(), y = Fq2::zero();
    if (lane < 6) {
        x = ldq(a + lane);
        if (K != 2) x = fq2_conj(x);
        const int e = 2 * (lane % 3) + lane / 3;       // exponent index 0..5
        typedef PairingConsts C;
        if (K == 2) {
            y = fq2_embed(e == 0 ? Fq::one() : e == 1 ? C::FROB2_1() : e == 2 ? C::FROB2_2() : e == 3 ? C::FROB2_3()
                          : e == 4 ? C::FROB2_4() : C::FROB2_5());
        } else if (K == 1) {
            y = e == 0 ? Fq2::one() : e == 1 ? Fq2{C::FROB1_1_C0(), C::FROB1_1_C1()} : e == 2 ? Fq2{C::FROB1_2_C0(), C::FROB1_2_C1()}
                : e == 3 ? Fq2{C::FROB1_3_C0(), C::FROB1_3_C1()} : e == 4 ? Fq2{C::FROB1_4_C0(), C::FROB1_4_C1()}
                         : Fq2{C::FROB1_5_C0(), C::FROB1_5_C1()};
        } else {
            y = e == 0 ? Fq2::one() : e == 1 ? Fq2{C::FROB3_1_C0(), C::FROB3_1_C1()} : e == 2 ? Fq2{C::FROB3_2_C0(), C::FROB3_2_C1()}
                : e == 3 ? Fq2{C::FROB3_3_C0(), C::FROB3_3_C1()} : e == 4 ? Fq2{C::FROB3_4_C0(), C::FROB3_4_C1()}
                         : Fq2{C::FROB3_5_C0(), C::FROB3_5_C1()};
        }
    }
    const Fq2 p = x * y;
    __syncwarp();
    if (lane < 6) stq(d + lane, p);
    __syncwarp();
}

// ---------------------------------------------------------------- inter-warp flags (shared memory)
__device__ __forceinline__ void flag_publish(int *flag, int v) {     // whole warp calls, after its last store
    __syncwarp();
    if (lane_id() == 0) {
        __threadfence_block();
        *reinterpret_cast<volatile int *>(flag) = v;
    }
}
__device__ __forceinline__ void flag_wait(const int *flag, int at_least) {
    if (lane_id() == 0) {
        // back off between polls: a spinning lane takes issue slots from the warp that shares its SM partition
        // (measured: a helper spinning beside the critical warp doubled that warp's time per product)
        while (*reinterpret_cast<const volatile int *>(flag) < at_least) __nanosleep(40);
        __threadfence_block();
    }
    __syncwarp();
}

// ---------------------------------------------------------------- the twist-point chain of one Miller loop
// Walks R over the NAF digits of 6x + 2 exactly as multi_miller_loop does and writes, per step, the line already scaled
// by the G1 point: (c0 * yP, c1 * xP, c2).  One product per lane and round; `*ready` counts finished lines.
struct LineState {
    Fq2 Rx, Ry, Rz, Qx, Qy, Qny, Q1x, Q1y, Q2x, Q2y;      // Qny = -Qy (negative NAF digits add -Q)
    Fq2 ey, ex;                       // (yP, 0), (xP, 0)
    Fq2 t[11];
};
__device__ __forceinline__ Fq2 g2_b_twist() {
    Fq2 b;
#pragma unroll
    for (int i = 0; i < 8; i++) { b.c0.l[i] = FqParams::G2B_C0(i); b.c1.l[i] = FqParams::G2B_C1(i); }
    return b;
}
// One round: every lane multiplies the operands it prepared; stores happen after all operand reads.
template <class Prep, class Store>
__device__ __forceinline__ void coop_round(Prep prep, Store store) {
    Fq2 x = Fq2::zero(), y = Fq2::zero();
    prep(x, y);
    const Fq2 p = x * y;
    __syncwarp();
    store(p);
    __syncwarp();
}
#define LZ_PREP [&](Fq2 & x, Fq2 & y)
#define LZ_STORE [&](const Fq2 &p)

__device__ __noinline__ void line_dbl(LineState *st, Fq2 *L) {
    const int lane = lane_id();
    Fq2 *t = st->t;
    // t0 = x y, t1 = b = y^2, t2 = c = z^2, t3 = (y + z)^2, t4 = j = x^2
    coop_round(LZ_PREP {
        if (lane < 5) {
            const Fq2 rx = ldq(&st->Rx), ry = ldq(&st->Ry), rz = ldq(&st->Rz);
            if (lane == 0) { x = rx; y = ry; }
            else if (lane == 1) { x = ry; y = ry; }
            else if (lane == 2) { x = rz; y = rz; }
            else if (lane == 3) { x = ry + rz; y = x; }
            else { x = rx; y = rx; }
        }
    }, LZ_STORE {
        if (lane < 5) stq(&t[lane], p);
    });
    // t5 = e = b' * 3c;  L0 = -h * yP with h = t3 - b - c;  L1 = 3j * xP
    coop_round(LZ_PREP {
        if (lane == 0) { x = g2_b_twist(); y = fq2_triple(ldq(&t[2])); }
        else if (lane == 1) { x = ldq(&t[1]) + ldq(&t[2]) - ldq(&t[3]); y = ldq(&st->ey); }
        else if (lane == 2) { x = fq2_triple(ldq(&t[4])); y = ldq(&st->ex); }
    }, LZ_STORE {
        if (lane == 0) stq(&t[5], p);
        else if (lane == 1) stq(L + 0, p);
        else if (lane == 2) stq(L + 1, p);
    });
    // X3 = a (b - f), t6 = g^2, t7 = e^2, Z3 = b h, L2 = i = e - b     (a = t0 / 2, f = 3e, g = (b + f) / 2)
    coop_round(LZ_PREP {
        if (lane < 5) {
            const Fq2 e = ldq(&t[5]), b = ldq(&t[1]);
            if (lane == 0) { x = fq2_half(ldq(&t[0])); y = b - fq2_triple(e); }
            else if (lane == 1) { x = fq2_half(b + fq2_triple(e)); y = x; }
            else if (lane == 2) { x = e; y = e; }
            else if (lane == 3) { x = b; y = ldq(&t[3]) - b - ldq(&t[2]); }
            else { x = e - b; y = Fq2::one(); }
        }
    }, LZ_STORE {
        if (lane == 0) stq(&st->Rx, p);
        else if (lane == 1) stq(&t[6], p);
        else if (lane == 2) stq(&t[7], p);
        else if (lane == 3) stq(&st->Rz, p);
        else if (lane == 4) stq(L + 2, p);
    });
    if (lane == 0) stq(&st->Ry, ldq(&t[6]) - fq2_triple(ldq(&t[7])));
    __syncwarp();
}
__device__ __noinline__ void line_add(LineState *st, const Fq2 *qx, const Fq2 *qy, Fq2 *L) {
    const int lane = lane_id();
    Fq2 *t = st->t;
    // t0 = qy z, t1 = qx z
    coop_round(LZ_PREP {
        if (lane < 2) { x = ldq(lane == 0 ? qy : qx); y = ldq(&st->Rz); }
    }, LZ_STORE {
        if (lane < 2) stq(&t[lane], p);
    });
    // theta = Ry - t0, lam = Rx - t1:  t2 = c = theta^2, t3 = d = lam^2, t4 = theta qx, t5 = lam qy,
    // L0 = lam * yP, L1 = -theta * xP
    coop_round(LZ_PREP {
        if (lane < 6) {
            const Fq2 th = ldq(&st->Ry) - ldq(&t[0]), lm = ldq(&st->Rx) - ldq(&t[1]);
            if (lane == 0) { x = th; y = th; }
            else if (lane == 1) { x = lm; y = lm; }
            else if (lane == 2) { x = th; y = ldq(qx); }
            else if (lane == 3) { x = lm; y = ldq(qy); }
            else if (lane == 4) { x = lm; y = ldq(&st->ey); }
            else { x = th.neg(); y = ldq(&st->ex); }
        }
    }, LZ_STORE {
        if (lane < 4) stq(&t[2 + lane], p);
        else if (lane < 6) stq(L + (lane - 4), p);
    });
    // t6 = e = lam d, t7 = f = z c, t8 = g = x d, L2 = t4 - t5
    coop_round(LZ_PREP {
        if (lane < 4) {
            const Fq2 lm = ldq(&st->Rx) - ldq(&t[1]);
            if (lane == 0) { x = lm; y = ldq(&t[3]); }
            else if (lane == 1) { x = ldq(&st->Rz); y = ldq(&t[2]); }
            else if (lane == 2) { x = ldq(&st->Rx); y = ldq(&t[3]); }
            else { x = ldq(&t[4]) - ldq(&t[5]); y = Fq2::one(); }
        }
    }, LZ_STORE {
        if (lane < 3) stq(&t[6 + lane], p);
        else if (lane == 3) stq(L + 2, p);
    });
    // h = e + f - 2g:  t9 = theta (g - h), t10 = e Ry, X3 = lam h, Z3 = z e
    coop_round(LZ_PREP {
        if (lane < 4) {
            const Fq2 e = ldq(&t[6]), g = ldq(&t[8]);
            const Fq2 h = e + ldq(&t[7]) - g.dbl();
            if (lane == 0) { x = ldq(&st->Ry) - ldq(&t[0]); y = g - h; }
            else if (lane == 1) { x = e; y = ldq(&st->Ry); }
            else if (lane == 2) { x = ldq(&st->Rx) - ldq(&t[1]); y = h; }
            else { x = ldq(&st->Rz); y = e; }
        }
    }, LZ_STORE {
        if (lane == 0) stq(&t[9], p);
        else if (lane == 1) stq(&t[10], p);
        else if (lane == 2) stq(&st->Rx, p);
        else if (lane == 3) stq(&st->Rz, p);
    });
    if (lane == 0) stq(&st->Ry, ldq(&t[9]) - ldq(&t[10]));
    __syncwarp();
}
// lines[3 n ..] for n = 0 .. kLines-1; *ready = n + 1 after line n.  P, Q neither at infinity.
__device__ __noinline__ void line_chain(LineState *st, const G1Affine &P, const G2Affine &Q, Fq2 *lines, int *ready) {
    const int lane = lane_id();
    if (lane == 0) {
        stq(&st->Rx, Q.x); stq(&st->Ry, Q.y); stq(&st->Rz, Fq2::one());
        stq(&st->Qx, Q.x); stq(&st->Qy, Q.y); stq(&st->Qny, Q.y.neg());
        stq(&st->ey, fq2_embed(P.y)); stq(&st->ex, fq2_embed(P.x));
    }
    __syncwarp();
    const Fq2 twx{PairingConsts::TW_X_C0(), PairingConsts::TW_X_C1()}, twy{PairingConsts::TW_Y_C0(), PairingConsts::TW_Y_C1()};
    // q1 = (conj(Qx) twx, conj(Qy) twy);  q2 = (conj(q1x) twx, -conj(q1y) twy)
    coop_round(LZ_PREP {
        if (lane == 0) { x = fq2_conj(Q.x); y = twx; }
        else if (lane == 1) { x = fq2_conj(Q.y); y = twy; }
    }, LZ_STORE {
        if (lane == 0) stq(&st->Q1x, p);
        else if (lane == 1) stq(&st->Q1y, p);
    });
    coop_round(LZ_PREP {
        if (lane == 0) { x = fq2_conj(ldq(&st->Q1x)); y = twx; }
        else if (lane == 1) { x = fq2_conj(ldq(&st->Q1y)); y = twy; }
    }, LZ_STORE {
        if (lane == 0) stq(&st->Q2x, p);
        else if (lane == 1) stq(&st->Q2y, p.neg());
    });
    int n = 0;
#pragma unroll 1
    for (int i = kAteTop; i >= 0; i--) {
        line_dbl(st, lines + 3 * n);
        flag_publish(ready, ++n);
        const int d = ate_digit(i);
        if (d) {
            line_add(st, &st->Qx, d > 0 ? &st->Qy : &st->Qny, lines + 3 * n);
            flag_publish(ready, ++n);
        }
    }
    line_add(st, &st->Q1x, &st->Q1y, lines + 3 * n);
    flag_publish(ready, ++n);
    line_add(st, &st->Q2x, &st->Q2y, lines + 3 * n);
    flag_publish(ready, ++n);
}

// ---------------------------------------------------------------- the f chain of one Miller loop
// SCALED: `lines` is the shared array a line_chain is filling (wait on *ready).  Otherwise `lines` are the PREPARED
// (unscaled) coefficients of a fixed G2 point in global memory; lanes 18..20 of the preceding product scale the next
// line by emb = {(yP, 0), (xP, 0), 1}.  Either way the line l0 + l1 w + l2 v w is handed to the product as a dense
// operand (l0, 0, 0, l1, l2, 0) in ln[2][6], whose other slots stay zero: ONE product body serves squarings and line
// products - a second (sparse) instantiation doubles the instruction footprint of a loop that runs on a lone warp.
// The loop runs the iterations i_hi .. i_lo of the bits of 6x + 2 starting from f = 1, then `tail_sq` bare squarings,
// then (final_lines) the two Frobenius lines.  The value of the whole loop factors as
//     f = (loop over 64 .. m, then m squarings) * (loop over m-1 .. 0 and the final lines, started from 1),
// so two warps can each run a share of the (A, B) loop (kMillerSplit): 97 + 97 products side by side instead of 152.
constexpr int kMillerSplit = 41;
LZ_HD constexpr int lines_before(int i_hi) {          // lines consumed by the iterations 63 .. i_hi + 1
    int c = 0;
    for (int i = kAteTop; i > i_hi; i--) c += 1 + (ate_digit(i) != 0 ? 1 : 0);
    return c;
}
template <bool SCALED>
__device__ __noinline__ void miller_f(Fq2 *f, const Fq2 *lines, const int *ready, Fq2 *ln, const Fq2 *emb, Scratch *s,
                                      int i_hi = kAteTop, int i_lo = 0, int tail_sq = 0, bool final_lines = true) {
    const int lane = lane_id();
    f12_set_one(f);
    int c = lines_before(i_hi), scaled = c;
    const int slot = lane % 3 == 0 ? 0 : 2 + lane % 3;          // coefficient index of line component lane % 3: 0, 3, 4
    auto step = [&](bool is_line) {
        const Fq2 *sa = nullptr, *sb = nullptr;
        Fq2 *so = nullptr;
        const Fq2 *b = f;
        if (SCALED) {
            if (is_line) {
                flag_wait(ready, c + 1);
                if (lane < 3) stq(ln + slot, ldq(lines + 3 * c + lane));
                __syncwarp();
                b = ln;
            }
        } else {
            if (is_line) b = ln + 6 * (c & 1);
            const int target = is_line ? c + 1 : c;
            if (scaled == target && target < kLines) {
                if (lane >= 18 && lane < 21) {
                    sa = lines + 3 * target + (lane - 18);
                    sb = emb + (lane - 18);
                    so = ln + 6 * (target & 1) + slot;
                }
                scaled++;
            }
        }
        f12_mul<false>(f, f, b, s, sa, sb, so);
        if (is_line) c++;
    };
#pragma unroll 1
    for (int i = i_hi; i >= i_lo; i--) {
        if (i != i_hi || !SCALED) step(false);      // f = 1 before the first iteration (prepared lines: the squaring of 1 carries the first scaling)
        step(true);
        if (ate_digit(i)) step(true);
    }
#pragma unroll 1
    for (int i = 0; i < tail_sq; i++) step(false);
    if (final_lines) {
        step(true);
        step(true);
    }
}

// ---------------------------------------------------------------- final exponentiation (pairing.cuh's chain)
// r = conj(a^x) for a in the cyclotomic subgroup.  a^x = product of a^(2^t) over the set bits t of x: THIS warp only
// squares (62 products) and hands every a^(2^t) with bit t set to a helper warp, which multiplies them up as they
// appear (27 products, finished one product after the last squaring): 63 products of latency instead of 89.
constexpr int kXBits = popcnt64(kBnX);               // 28
struct ExpShare {
    Fq2 *items;          // kXBits Fq12 values
    Fq2 *prod;           // the helper's running product
    int *count, *done;   // items published so far (all exponentiations of a proof), exponentiations finished
};
__device__ __noinline__ void f12_exp_neg_x(Fq2 *r, const Fq2 *a, Fq2 *q, Scratch *s, const ExpShare &sh, int gen) {
    int j = 0;
#pragma unroll 1
    for (int t = 0; t < 63; t++) {
        if (t == 0) f12_copy(q, a);
        else f12_mul<false>(q, q, q, s);
        if ((kBnX >> t) & 1ull) {
            f12_copy(sh.items + 6 * j, q);
            j++;
            flag_publish(sh.count, gen * kXBits + j);
        }
    }
    flag_wait(sh.done, gen + 1);
    f12_conj(r, sh.prod);
}
// the helper warp's side of exponentiation number `gen` of a proof
__device__ __noinline__ void f12_exp_helper(Scratch *s, const ExpShare &sh, int gen) {
    flag_wait(sh.count, gen * kXBits + 1);
    f12_copy(sh.prod, sh.items);
#pragma unroll 1
    for (int j = 1; j < kXBits; j++) {
        flag_wait(sh.count, gen * kXBits + j + 1);
        f12_mul<false>(sh.prod, sh.prod, sh.items + 6 * j, s);
    }
    flag_publish(sh.done, gen + 1);
}
// out = f^((p^12 - 1)/r * c) as final_exponentiation computes it; T: ten Fq12 slots of scratch (60 Fq2); out may be f.
// A helper warp must run f12_exp_helper(.., sh, 0 .. 2) beside it.
__device__ __noinline__ void final_exp(Fq2 *out, const Fq2 *f, Fq2 *T, Scratch *s, const ExpShare &sh) {
    const int lane = lane_id();
    Fq2 *R = T + 6 * 8, *X = T + 6 * 9, *S0 = T, *S1 = T + 6, *S2 = T + 12, *S4 = T + 24, *S5 = T + 30, *S6 = T + 36, *S7 = T + 42;
    // easy part: r = conj(f) / f = conj(f)^2 / N with N = f conj(f) in Fq6
    f12_conj(S0, f);
    f12_mul<false>(S1, S0, f, s);                       // (N, 0)
    if (lane == 0) {
        Fq6 *n = reinterpret_cast<Fq6 *>(S1);
        f6_inv(*n, *n);
    }
    __syncwarp();
    f12_mul<false>(S2, S0, S1, s);                      // 1 / f
    f12_mul<false>(R, S0, S2, s);                       // f^(p^6 - 1)
    f12_frob<2>(S0, R);
    f12_mul<false>(R, S0, R, s);                        // ^(p^2 + 1)
    // hard part
    f12_exp_neg_x(S0, R, S7, s, sh, 0);                 // y0
    f12_mul<false>(S1, S0, S0, s);                      // y1 = y0^2
    f12_mul<false>(S2, S1, S1, s);                      // y2
    f12_mul<false>(S2, S2, S1, s);                      // y3
    f12_exp_neg_x(S4, S2, S7, s, sh, 1);                // y4
    f12_mul<false>(S5, S4, S4, s);                      // y5
    f12_exp_neg_x(S6, S5, S7, s, sh, 2);                // y6
    f12_conj(S2, S2);
    f12_conj(S6, S6);
    f12_mul<false>(S6, S6, S4, s);                      // y7
    f12_mul<false>(S6, S6, S2, s);                      // y8
    f12_mul<false>(S1, S6, S1, s);                      // y9
    f12_mul<false>(S4, S6, S4, s);                      // y10
    f12_mul<false>(S4, S4, R, s);                       // y11
    f12_frob<1>(S0, S1);                                // y12
    f12_mul<false>(S0, S0, S4, s);                      // y13
    f12_frob<2>(S5, S6);
    f12_mul<false>(S0, S5, S0, s);                      // y14
    f12_conj(S5, R);
    f12_mul<false>(S5, S5, S1, s);                      // y15
    f12_frob<3>(X, S5);
    f12_mul<false>(out, X, S0, s);
}
__device__ __forceinline__ bool f12_equal(const Fq2 *a, const Fq2 *b) {     // whole warp; a, b anywhere
    const int lane = lane_id();
    bool eq = true;
    if (lane < 6) eq = ldq(a + lane) == ldq(b + lane);
    return __all_sync(0xffffffffu, eq);
}

// ---------------------------------------------------------------- G2 ladder for the r-torsion test of B
struct LadderState {
    Fq2 X, Y, ZZ, ZZZ, bx, by;
    Fq2 t[8];
};
__device__ __noinline__ void ladder_dbl(LadderState *st) {          // XYZZ dbl-2008-s-1, three rounds; point not special
    const int lane = lane_id();
    Fq2 *t = st->t;
    // t0 = V = (2Y)^2, t1 = X^2
    coop_round(LZ_PREP {
        if (lane == 0) { x = ldq(&st->Y).dbl(); y = x; }
        else if (lane == 1) { x = ldq(&st->X); y = x; }
    }, LZ_STORE {
        if (lane < 2) stq(&t[lane], p);
    });
    // t2 = W = U V, t3 = S = X V, t4 = M^2 (M = 3 t1), ZZ = V ZZ
    coop_round(LZ_PREP {
        if (lane < 4) {
            const Fq2 V = ldq(&t[0]);
            if (lane == 0) { x = ldq(&st->Y).dbl(); y = V; }
            else if (lane == 1) { x = ldq(&st->X); y = V; }
            else if (lane == 2) { x = fq2_triple(ldq(&t[1])); y = x; }
            else { x = V; y = ldq(&st->ZZ); }
        }
    }, LZ_STORE {
        if (lane < 3) stq(&t[2 + lane], p);
        else if (lane == 3) stq(&st->ZZ, p);
    });
    // X3 = t4 - 2S;  t5 = M (S - X3), t6 = W Y, ZZZ = W ZZZ
    coop_round(LZ_PREP {
        if (lane < 3) {
            const Fq2 W = ldq(&t[2]);
            if (lane == 0) { const Fq2 S = ldq(&t[3]); x = fq2_triple(ldq(&t[1])); y = S - (ldq(&t[4]) - S.dbl()); }
            else if (lane == 1) { x = W; y = ldq(&st->Y); }
            else { x = W; y = ldq(&st->ZZZ); }
        }
    }, LZ_STORE {
        if (lane == 0) stq(&t[5], p);
        else if (lane == 1) stq(&t[6], p);
        else if (lane == 2) stq(&st->ZZZ, p);
    });
    if (lane == 0) {
        stq(&st->X, ldq(&t[4]) - ldq(&t[3]).dbl());
        stq(&st->Y, ldq(&t[5]) - ldq(&t[6]));
    }
    __syncwarp();
}
// acc += (bx, by), madd-2008-s, four rounds.  Returns false (state untouched) when the addition is special
// (acc == +-B): the caller then takes the serial formulas.
__device__ __noinline__ bool ladder_madd(LadderState *st) {
    const int lane = lane_id();
    Fq2 *t = st->t;
    // t0 = U2 = bx ZZ, t1 = S2 = by ZZZ
    coop_round(LZ_PREP {
        if (lane < 2) { x = ldq(lane == 0 ? &st->bx : &st->by); y = ldq(lane == 0 ? &st->ZZ : &st->ZZZ); }
    }, LZ_STORE {
        if (lane < 2) stq(&t[lane], p);
    });
    bool special = false;
    if (lane == 0) special = (ldq(&t[0]) - ldq(&st->X)).is_zero();
    if (__shfl_sync(0xffffffffu, (int)special, 0)) return false;
    // Pp = U2 - X, R = S2 - Y:  t2 = PP = Pp^2, t3 = R^2
    coop_round(LZ_PREP {
        if (lane == 0) { x = ldq(&t[0]) - ldq(&st->X); y = x; }
        else if (lane == 1) { x = ldq(&t[1]) - ldq(&st->Y); y = x; }
    }, LZ_STORE {
        if (lane < 2) stq(&t[2 + lane], p);
    });
    // t4 = PPP = Pp PP, t5 = Q = X PP, ZZ = ZZ PP
    coop_round(LZ_PREP {
        if (lane < 3) {
            const Fq2 PP = ldq(&t[2]);
            if (lane == 0) { x = ldq(&t[0]) - ldq(&st->X); y = PP; }
            else if (lane == 1) { x = ldq(&st->X); y = PP; }
            else { x = ldq(&st->ZZ); y = PP; }
        }
    }, LZ_STORE {
        if (lane == 0) stq(&t[4], p);
        else if (lane == 1) stq(&t[5], p);
        else if (lane == 2) stq(&st->ZZ, p);
    });
    // X3 = t3 - PPP - 2Q;  t6 = R (Q - X3), t7 = Y PPP, ZZZ = ZZZ PPP
    coop_round(LZ_PREP {
        if (lane < 3) {
            const Fq2 PPP = ldq(&t[4]);
            if (lane == 0) { const Fq2 Q = ldq(&t[5]); x = ldq(&t[1]) - ldq(&st->Y); y = Q - (ldq(&t[3]) - PPP - Q.dbl()); }
            else if (lane == 1) { x = ldq(&st->Y); y = PPP; }
            else { x = ldq(&st->ZZZ); y = PPP; }
        }
    }, LZ_STORE {
        if (lane == 0) stq(&t[6], p);
        else if (lane == 1) stq(&t[7], p);
        else if (lane == 2) stq(&st->ZZZ, p);
    });
    if (lane == 0) {
        stq(&st->X, ldq(&t[3]) - ldq(&t[4]) - ldq(&t[5]).dbl());
        stq(&st->Y, ldq(&t[6]) - ldq(&t[7]));
    }
    __syncwarp();
    return true;
}
// One bit of the ladder: acc = 2 acc, then acc += (bx, by) when `add`.  Special points (acc at infinity or of order two,
// acc == +-B) take the complete serial formulas on lane 0.
__device__ __forceinline__ void ladder_step(LadderState *st, bool add) {
    const int lane = lane_id();
    auto serial = [&](bool add) {          // special points: the complete formulas on one lane
        if (lane == 0) {
            G2XYZZ a{ldq(&st->X), ldq(&st->Y), ldq(&st->ZZ), ldq(&st->ZZZ)};
            if (add) a.madd_cold(G2Affine{ldq(&st->bx), ldq(&st->by)});
            else a.dbl_cold();
            stq(&st->X, a.x); stq(&st->Y, a.y); stq(&st->ZZ, a.zz); stq(&st->ZZZ, a.zzz);
        }
        __syncwarp();
    };
    auto is_special = [&]() {              // infinity or a point of order two
        bool sp = false;
        if (lane == 0) sp = ldq(&st->ZZ).is_zero() || ldq(&st->Y).is_zero();
        return __shfl_sync(0xffffffffu, (int)sp, 0) != 0;
    };
    if (is_special()) serial(false);
    else ladder_dbl(st);
    if (add) {
        if (is_special() || !ladder_madd(st)) serial(true);
    }
}
// B (on the twist, not infinity) in the r-torsion subgroup?  The ladder computes [x] B (62 doublings, 27 additions with
// their independent products on different lanes); lane 0 then finishes the test of pairing.cuh g2_subgroup_from_xp.
__device__ __noinline__ bool g2_in_subgroup(LadderState *st, const G2Affine &B) {
    const int lane = lane_id();
    if (lane == 0) {
        stq(&st->X, B.x); stq(&st->Y, B.y); stq(&st->ZZ, Fq2::one()); stq(&st->ZZZ, Fq2::one());
        stq(&st->bx, B.x); stq(&st->by, B.y);
    }
    __syncwarp();
#pragma unroll 1
    for (int i = 61; i >= 0; i--) ladder_step(st, ((kBnX >> i) & 1ull) != 0);     // bit 62 is the leading one of x
    bool ok = false;
    if (lane == 0) ok = g2_subgroup_from_xp(B, G2XYZZ{ldq(&st->X), ldq(&st->Y), ldq(&st->ZZ), ldq(&st->ZZZ)});
    return __shfl_sync(0xffffffffu, (int)ok, 0) != 0;
}

// ---------------------------------------------------------------- vk_x from the byte-window tables
// tab[((i * 32 + w) * 255 + d - 1)] = d * 256^w * gamma_abc[i + 1].  x: the proof's n_pub canonical scalars (32 LE
// bytes each).  Whole warp; the affine result is returned on every lane.
__device__ __noinline__ G1Affine vkx_from_tables(const G1Affine *__restrict__ tab, const G1Affine *__restrict__ gamma_abc,
                                                 const uint8_t *__restrict__ x, uint32_t n_pub) {
    const int lane = lane_id();
    G1XYZZ acc = G1XYZZ::inf();
    const uint32_t pairs = n_pub * kTabWindows;
#pragma unroll 1
    for (uint32_t q0 = 0; q0 < pairs; q0 += 32) {               // window-major: small scalars fill whole steps
        const uint32_t q = q0 + lane;
        uint32_t d = 0, i = 0, w = 0;
        if (q < pairs) { w = q / n_pub; i = q - w * n_pub; d = x[(size_t)i * 32 + w]; }
        if (__ballot_sync(0xffffffffu, d != 0) == 0) continue;
        if (d) acc.madd(ldg_vec(tab + ((size_t)i * kTabWindows + w) * kTabDigits + (d - 1)));
    }
#pragma unroll 1
    for (int off = 16; off > 0; off >>= 1) {
        G1XYZZ o;
        uint32_t *ow = reinterpret_cast<uint32_t *>(&o);
        const uint32_t *aw = reinterpret_cast<const uint32_t *>(&acc);
#pragma unroll
        for (int k = 0; k < (int)(sizeof(G1XYZZ) / 4); k++) ow[k] = __shfl_down_sync(0xffffffffu, aw[k], off);
        acc.add_cold(o);
    }
    G1Affine r = G1Affine::inf();
    if (lane == 0) {
        acc.madd_cold(ldg_vec(gamma_abc));
        r = acc.to_affine();
    }
    uint32_t *rw = reinterpret_cast<uint32_t *>(&r);
#pragma unroll
    for (int k = 0; k < (int)(sizeof(G1Affine) / 4); k++) rw[k] = __shfl_sync(0xffffffffu, rw[k], 0);
    return r;
}

}  // namespace coop
}  // namespace lzkp
