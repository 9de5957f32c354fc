// Device-only carry-chain field arithmetic (PTX add.cc / mad.lo.cc / madc.hi.cc), N = 4 and 8 limbs.
//
// Montgomery product, row-wise (CIOS) with TWO interleaved accumulators so that every 32x32->64
// partial product lands on an aligned (lo, hi) register pair and one carry chain runs over the
// pairs — ptxas turns each mad.lo.cc / madc.hi.cc pair into one IMAD.WIDE.U32(.X):
//     E[j] sits at limb position j,  O[j] at position j + 1
//     even-index limbs x[0], x[2], ... multiply into the pairs (E[1]:E[0]), (E[3]:E[2]), ...
//     odd-index  limbs x[1], x[3], ... multiply into the pairs (O[1]:O[0]), (O[3]:O[2]), ...
// After a row (T += a*b_i; m = T[0]*n0inv; T += p*m) limb 0 is zero and T is shifted down one limb:
// O becomes the new E, E[2..] becomes the new O, E[1] is folded into the new E[0] and its carry
// rides into the new O chain; the chains' carry-outs become the top limbs of the new O.
// Works for every odd p < 2^(32N) (the value may transiently need N+1 limbs; the final conditional
// subtraction takes the top carry).  Checked bit-for-bit against fe_mont_mul_portable by
// tests/test_gpu_field.py (zkb_debug_field_ops) and by every GPU parity test.
#pragma once
#include "field.cuh"

#if defined(__CUDA_ARCH__) && !defined(ZKB_NO_PTX_FIELD)
#define ZKB_FIELD_PTX 1
// accumulator operands of the chains: early-clobber (see the note above mad_chain4); -DZKB_NO_EARLY_CLOBBER for the A/B only —
// the lazy-reduction code is wrong without it
#ifdef ZKB_NO_EARLY_CLOBBER
#define ZKB_ACC_C "+r"
#else
#define ZKB_ACC_C "+&r"
#endif
#define ZKB_ACC(x) ZKB_ACC_C(x)

namespace zkb {

// ---- N = 8: four (lo, hi) pairs per chain ---------------------------------------------------
// acc pairs = x_k * y   (no accumulate: first row)
__device__ __forceinline__ void mul_pairs4(uint32_t* acc, uint32_t x0, uint32_t x1, uint32_t x2, uint32_t x3, uint32_t y) {
    asm("mul.lo.u32 %0, %8, %12;\n\t"
        "mul.hi.u32 %1, %8, %12;\n\t"
        "mul.lo.u32 %2, %9, %12;\n\t"
        "mul.hi.u32 %3, %9, %12;\n\t"
        "mul.lo.u32 %4, %10, %12;\n\t"
        "mul.hi.u32 %5, %10, %12;\n\t"
        "mul.lo.u32 %6, %11, %12;\n\t"
        "mul.hi.u32 %7, %11, %12;"
        : "=r"(acc[0]), "=r"(acc[1]), "=r"(acc[2]), "=r"(acc[3]), "=r"(acc[4]), "=r"(acc[5]), "=r"(acc[6]), "=r"(acc[7])
        : "r"(x0), "r"(x1), "r"(x2), "r"(x3), "r"(y));
}

// (the accumulator operands are early-clobber: a chain writes acc[0] before it reads its last inputs, and the compiler would
// otherwise let an accumulator limb and an input that hold the same value - two literal zeros, say - share one register)
// acc pairs += x_k * y with one carry chain; returns cin + the carry out of the top pair (cin: the carries this limb
// position has already collected in this row, so that two chains into the same accumulator need no separate addition)
__device__ __forceinline__ uint32_t mad_chain4(uint32_t* acc, uint32_t x0, uint32_t x1, uint32_t x2, uint32_t x3, uint32_t y,
                                               uint32_t cin = 0) {
    uint32_t c;
    asm("mad.lo.cc.u32 %0, %9, %13, %0;\n\t"
        "madc.hi.cc.u32 %1, %9, %13, %1;\n\t"
        "madc.lo.cc.u32 %2, %10, %13, %2;\n\t"
        "madc.hi.cc.u32 %3, %10, %13, %3;\n\t"
        "madc.lo.cc.u32 %4, %11, %13, %4;\n\t"
        "madc.hi.cc.u32 %5, %11, %13, %5;\n\t"
        "madc.lo.cc.u32 %6, %12, %13, %6;\n\t"
        "madc.hi.cc.u32 %7, %12, %13, %7;\n\t"
        "addc.u32 %8, %14, 0;"
        : ZKB_ACC(acc[0]), ZKB_ACC(acc[1]), ZKB_ACC(acc[2]), ZKB_ACC(acc[3]), ZKB_ACC(acc[4]), ZKB_ACC(acc[5]), ZKB_ACC(acc[6]), ZKB_ACC(acc[7]), "=r"(c)
        : "r"(x0), "r"(x1), "r"(x2), "r"(x3), "r"(y), "r"(cin));
    return c;
}

// e0 = f0 + f1 (the folded limb), its carry continues into:  acc pairs += x_k * y ; returns carry out
__device__ __forceinline__ uint32_t mad_chain4_fold(uint32_t& e0, uint32_t f0, uint32_t f1, uint32_t* acc, uint32_t x0, uint32_t x1,
                                                    uint32_t x2, uint32_t x3, uint32_t y) {
    uint32_t c;
    asm("add.cc.u32 %9, %10, %11;\n\t"
        "madc.lo.cc.u32 %0, %12, %16, %0;\n\t"
        "madc.hi.cc.u32 %1, %12, %16, %1;\n\t"
        "madc.lo.cc.u32 %2, %13, %16, %2;\n\t"
        "madc.hi.cc.u32 %3, %13, %16, %3;\n\t"
        "madc.lo.cc.u32 %4, %14, %16, %4;\n\t"
        "madc.hi.cc.u32 %5, %14, %16, %5;\n\t"
        "madc.lo.cc.u32 %6, %15, %16, %6;\n\t"
        "madc.hi.cc.u32 %7, %15, %16, %7;\n\t"
        "addc.u32 %8, 0, 0;"
        : ZKB_ACC(acc[0]), ZKB_ACC(acc[1]), ZKB_ACC(acc[2]), ZKB_ACC(acc[3]), ZKB_ACC(acc[4]), ZKB_ACC(acc[5]), ZKB_ACC(acc[6]), ZKB_ACC(acc[7]), "=r"(c),
          "=r"(e0)
        : "r"(f0), "r"(f1), "r"(x0), "r"(x1), "r"(x2), "r"(x3), "r"(y));
    return c;
}

// acc pairs += x_k * y with a carry-in at the BOTTOM of the chain (cbot in {0, 1}: the carry of a fold done outside); returns
// the carry out of the top pair
__device__ __forceinline__ uint32_t mad_chain4_cbot(uint32_t* acc, uint32_t x0, uint32_t x1, uint32_t x2, uint32_t x3, uint32_t y,
                                                    uint32_t cbot) {
    uint32_t c, t;
    asm("add.cc.u32 %9, %15, 0xFFFFFFFF;\n\t"
        "madc.lo.cc.u32 %0, %10, %14, %0;\n\t"
        "madc.hi.cc.u32 %1, %10, %14, %1;\n\t"
        "madc.lo.cc.u32 %2, %11, %14, %2;\n\t"
        "madc.hi.cc.u32 %3, %11, %14, %3;\n\t"
        "madc.lo.cc.u32 %4, %12, %14, %4;\n\t"
        "madc.hi.cc.u32 %5, %12, %14, %5;\n\t"
        "madc.lo.cc.u32 %6, %13, %14, %6;\n\t"
        "madc.hi.cc.u32 %7, %13, %14, %7;\n\t"
        "addc.u32 %8, 0, 0;"
        : ZKB_ACC(acc[0]), ZKB_ACC(acc[1]), ZKB_ACC(acc[2]), ZKB_ACC(acc[3]), ZKB_ACC(acc[4]), ZKB_ACC(acc[5]), ZKB_ACC(acc[6]), ZKB_ACC(acc[7]), "=r"(c), "=r"(t)
        : "r"(x0), "r"(x1), "r"(x2), "r"(x3), "r"(y), "r"(cbot));
    return c;
}

// The reduction chains of fe_mont_mul_low64 (p mod 2^64 = 2^64 - 2^32 + 1, m = -acc[0] mod 2^32): the bottom pair's product
// is not multiplied.
// even: acc pairs += (0 : m) + x1 * y << 64 + x2 * y << 128 + x3 * y << 192 with p0 = 1, i.e. the bottom pair gets m.  acc[0] + m
// = 0 mod 2^32 carries exactly when acc[0] != 0; acc[0] itself (which would become 0) is left as it is: the shift drops it.
// Returns cin + the carry out of the top pair.
__device__ __forceinline__ uint32_t mad_chain4_low_even(uint32_t* acc, uint32_t x1, uint32_t x2, uint32_t x3, uint32_t y, uint32_t cin) {
    uint32_t c, t;
    asm("add.cc.u32 %8, %9, 0xFFFFFFFF;\n\t"
        "addc.cc.u32 %0, %0, 0;\n\t"
        "madc.lo.cc.u32 %1, %10, %13, %1;\n\t"
        "madc.hi.cc.u32 %2, %10, %13, %2;\n\t"
        "madc.lo.cc.u32 %3, %11, %13, %3;\n\t"
        "madc.hi.cc.u32 %4, %11, %13, %4;\n\t"
        "madc.lo.cc.u32 %5, %12, %13, %5;\n\t"
        "madc.hi.cc.u32 %6, %12, %13, %6;\n\t"
        "addc.u32 %7, %14, 0;"
        : ZKB_ACC(acc[1]), ZKB_ACC(acc[2]), ZKB_ACC(acc[3]), ZKB_ACC(acc[4]), ZKB_ACC(acc[5]), ZKB_ACC(acc[6]), ZKB_ACC(acc[7]), "=r"(c), "=r"(t)
        : "r"(acc[0]), "r"(x1), "r"(x2), "r"(x3), "r"(y), "r"(cin));
    return c;
}
// odd: acc pairs += (hi : lo) + x1 * y << 64 + x2 * y << 128 + x3 * y << 192, where (hi : lo) = p1 * m = m 2^32 - m as a
// 64-bit pair (p1 = 2^32 - 1): lo = -m = the row's T0, hi = m - [m != 0].  Returns cin + the carry out of the top pair.
__device__ __forceinline__ uint32_t mad_chain4_low_odd(uint32_t* acc, uint32_t lo, uint32_t hi, uint32_t x1, uint32_t x2, uint32_t x3,
                                                       uint32_t y, uint32_t cin) {
    uint32_t c;
    asm("add.cc.u32 %0, %0, %9;\n\t"
        "addc.cc.u32 %1, %1, %10;\n\t"
        "madc.lo.cc.u32 %2, %11, %14, %2;\n\t"
        "madc.hi.cc.u32 %3, %11, %14, %3;\n\t"
        "madc.lo.cc.u32 %4, %12, %14, %4;\n\t"
        "madc.hi.cc.u32 %5, %12, %14, %5;\n\t"
        "madc.lo.cc.u32 %6, %13, %14, %6;\n\t"
        "madc.hi.cc.u32 %7, %13, %14, %7;\n\t"
        "addc.u32 %8, %15, 0;"
        : ZKB_ACC(acc[0]), ZKB_ACC(acc[1]), ZKB_ACC(acc[2]), ZKB_ACC(acc[3]), ZKB_ACC(acc[4]), ZKB_ACC(acc[5]), ZKB_ACC(acc[6]), ZKB_ACC(acc[7]), "=r"(c)
        : "r"(lo), "r"(hi), "r"(x1), "r"(x2), "r"(x3), "r"(y), "r"(cin));
    return c;
}
// m = -t0 mod 2^32 (the row's multiplier when n0inv = 2^32 - 1) and mh = m - [m != 0]: sub.cc borrows exactly when t0 != 0
__device__ __forceinline__ void low64_m(uint32_t& m, uint32_t& mh, uint32_t t0) {
    asm("sub.cc.u32 %0, 0, %2;\n\t"
        "subc.u32 %1, %0, 0;"
        : "=r"(m), "=r"(mh)
        : "r"(t0));
}

// ---- N = 4: two pairs per chain --------------------------------------------------------------
__device__ __forceinline__ uint32_t mad_chain2_cbot(uint32_t* acc, uint32_t x0, uint32_t x1, uint32_t y, uint32_t cbot) {
    uint32_t c, t;
    asm("add.cc.u32 %5, %9, 0xFFFFFFFF;\n\t"
        "madc.lo.cc.u32 %0, %6, %8, %0;\n\t"
        "madc.hi.cc.u32 %1, %6, %8, %1;\n\t"
        "madc.lo.cc.u32 %2, %7, %8, %2;\n\t"
        "madc.hi.cc.u32 %3, %7, %8, %3;\n\t"
        "addc.u32 %4, 0, 0;"
        : ZKB_ACC(acc[0]), ZKB_ACC(acc[1]), ZKB_ACC(acc[2]), ZKB_ACC(acc[3]), "=r"(c), "=r"(t)
        : "r"(x0), "r"(x1), "r"(y), "r"(cbot));
    return c;
}
__device__ __forceinline__ void mul_pairs2(uint32_t* acc, uint32_t x0, uint32_t x1, uint32_t y) {
    asm("mul.lo.u32 %0, %4, %6;\n\t"
        "mul.hi.u32 %1, %4, %6;\n\t"
        "mul.lo.u32 %2, %5, %6;\n\t"
        "mul.hi.u32 %3, %5, %6;"
        : "=r"(acc[0]), "=r"(acc[1]), "=r"(acc[2]), "=r"(acc[3])
        : "r"(x0), "r"(x1), "r"(y));
}
__device__ __forceinline__ uint32_t mad_chain2(uint32_t* acc, uint32_t x0, uint32_t x1, uint32_t y, uint32_t cin = 0) {
    uint32_t c;
    asm("mad.lo.cc.u32 %0, %5, %7, %0;\n\t"
        "madc.hi.cc.u32 %1, %5, %7, %1;\n\t"
        "madc.lo.cc.u32 %2, %6, %7, %2;\n\t"
        "madc.hi.cc.u32 %3, %6, %7, %3;\n\t"
        "addc.u32 %4, %8, 0;"
        : ZKB_ACC(acc[0]), ZKB_ACC(acc[1]), ZKB_ACC(acc[2]), ZKB_ACC(acc[3]), "=r"(c)
        : "r"(x0), "r"(x1), "r"(y), "r"(cin));
    return c;
}
__device__ __forceinline__ uint32_t mad_chain2_fold(uint32_t& e0, uint32_t f0, uint32_t f1, uint32_t* acc, uint32_t x0, uint32_t x1,
                                                    uint32_t y) {
    uint32_t c;
    asm("add.cc.u32 %5, %6, %7;\n\t"
        "madc.lo.cc.u32 %0, %8, %10, %0;\n\t"
        "madc.hi.cc.u32 %1, %8, %10, %1;\n\t"
        "madc.lo.cc.u32 %2, %9, %10, %2;\n\t"
        "madc.hi.cc.u32 %3, %9, %10, %3;\n\t"
        "addc.u32 %4, 0, 0;"
        : ZKB_ACC(acc[0]), ZKB_ACC(acc[1]), ZKB_ACC(acc[2]), ZKB_ACC(acc[3]), "=r"(c), "=r"(e0)
        : "r"(f0), "r"(f1), "r"(x0), "r"(x1), "r"(y));
    return c;
}

// ---- additions / conditional subtraction as single carry chains -------------------------------------
// d = (carry:a) - p over N+1 limbs; the top limb is 0 when the difference is non-negative (then r = d), all ones otherwise
__device__ __forceinline__ void cond_sub_chain8(uint32_t* r, const uint32_t* a, uint32_t carry, const uint32_t* p) {
    uint32_t d[8], top;
    asm("sub.cc.u32 %0, %9, %17;\n\t"
        "subc.cc.u32 %1, %10, %18;\n\t"
        "subc.cc.u32 %2, %11, %19;\n\t"
        "subc.cc.u32 %3, %12, %20;\n\t"
        "subc.cc.u32 %4, %13, %21;\n\t"
        "subc.cc.u32 %5, %14, %22;\n\t"
        "subc.cc.u32 %6, %15, %23;\n\t"
        "subc.cc.u32 %7, %16, %24;\n\t"
        "subc.u32 %8, %25, 0;"
        : "=r"(d[0]), "=r"(d[1]), "=r"(d[2]), "=r"(d[3]), "=r"(d[4]), "=r"(d[5]), "=r"(d[6]), "=r"(d[7]), "=r"(top)
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(a[4]), "r"(a[5]), "r"(a[6]), "r"(a[7]), "r"(p[0]), "r"(p[1]), "r"(p[2]),
          "r"(p[3]), "r"(p[4]), "r"(p[5]), "r"(p[6]), "r"(p[7]), "r"(carry));
    const bool use_d = top == 0;
#pragma unroll
    for (int i = 0; i < 8; i++) r[i] = use_d ? d[i] : a[i];
}
__device__ __forceinline__ void cond_sub_chain4(uint32_t* r, const uint32_t* a, uint32_t carry, const uint32_t* p) {
    uint32_t d[4], top;
    asm("sub.cc.u32 %0, %5, %9;\n\t"
        "subc.cc.u32 %1, %6, %10;\n\t"
        "subc.cc.u32 %2, %7, %11;\n\t"
        "subc.cc.u32 %3, %8, %12;\n\t"
        "subc.u32 %4, %13, 0;"
        : "=r"(d[0]), "=r"(d[1]), "=r"(d[2]), "=r"(d[3]), "=r"(top)
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(p[0]), "r"(p[1]), "r"(p[2]), "r"(p[3]), "r"(carry));
    const bool use_d = top == 0;
#pragma unroll
    for (int i = 0; i < 4; i++) r[i] = use_d ? d[i] : a[i];
}
// s = a + b, returns the carry out
__device__ __forceinline__ uint32_t add_chain8(uint32_t* s, const uint32_t* a, const uint32_t* b) {
    uint32_t c;
    asm("add.cc.u32 %0, %9, %17;\n\t"
        "addc.cc.u32 %1, %10, %18;\n\t"
        "addc.cc.u32 %2, %11, %19;\n\t"
        "addc.cc.u32 %3, %12, %20;\n\t"
        "addc.cc.u32 %4, %13, %21;\n\t"
        "addc.cc.u32 %5, %14, %22;\n\t"
        "addc.cc.u32 %6, %15, %23;\n\t"
        "addc.cc.u32 %7, %16, %24;\n\t"
        "addc.u32 %8, 0, 0;"
        : "=r"(s[0]), "=r"(s[1]), "=r"(s[2]), "=r"(s[3]), "=r"(s[4]), "=r"(s[5]), "=r"(s[6]), "=r"(s[7]), "=r"(c)
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(a[4]), "r"(a[5]), "r"(a[6]), "r"(a[7]), "r"(b[0]), "r"(b[1]), "r"(b[2]),
          "r"(b[3]), "r"(b[4]), "r"(b[5]), "r"(b[6]), "r"(b[7]));
    return c;
}
__device__ __forceinline__ uint32_t add_chain4(uint32_t* s, const uint32_t* a, const uint32_t* b) {
    uint32_t c;
    asm("add.cc.u32 %0, %5, %9;\n\t"
        "addc.cc.u32 %1, %6, %10;\n\t"
        "addc.cc.u32 %2, %7, %11;\n\t"
        "addc.cc.u32 %3, %8, %12;\n\t"
        "addc.u32 %4, 0, 0;"
        : "=r"(s[0]), "=r"(s[1]), "=r"(s[2]), "=r"(s[3]), "=r"(c)
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]), "r"(b[2]), "r"(b[3]));
    return c;
}

// s = a + b + cin (cin in {0, 1}), returns the carry out: the upper half of a 2N-limb addition
__device__ __forceinline__ uint32_t add_chain8_cin(uint32_t* s, const uint32_t* a, const uint32_t* b, uint32_t cin) {
    uint32_t c, t;
    asm("add.cc.u32 %9, %26, 0xFFFFFFFF;\n\t"
        "addc.cc.u32 %0, %10, %18;\n\t"
        "addc.cc.u32 %1, %11, %19;\n\t"
        "addc.cc.u32 %2, %12, %20;\n\t"
        "addc.cc.u32 %3, %13, %21;\n\t"
        "addc.cc.u32 %4, %14, %22;\n\t"
        "addc.cc.u32 %5, %15, %23;\n\t"
        "addc.cc.u32 %6, %16, %24;\n\t"
        "addc.cc.u32 %7, %17, %25;\n\t"
        "addc.u32 %8, 0, 0;"
        : "=r"(s[0]), "=r"(s[1]), "=r"(s[2]), "=r"(s[3]), "=r"(s[4]), "=r"(s[5]), "=r"(s[6]), "=r"(s[7]), "=r"(c), "=r"(t)
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(a[4]), "r"(a[5]), "r"(a[6]), "r"(a[7]), "r"(b[0]), "r"(b[1]), "r"(b[2]),
          "r"(b[3]), "r"(b[4]), "r"(b[5]), "r"(b[6]), "r"(b[7]), "r"(cin));
    return c;
}
__device__ __forceinline__ uint32_t add_chain4_cin(uint32_t* s, const uint32_t* a, const uint32_t* b, uint32_t cin) {
    uint32_t c, t;
    asm("add.cc.u32 %5, %14, 0xFFFFFFFF;\n\t"
        "addc.cc.u32 %0, %6, %10;\n\t"
        "addc.cc.u32 %1, %7, %11;\n\t"
        "addc.cc.u32 %2, %8, %12;\n\t"
        "addc.cc.u32 %3, %9, %13;\n\t"
        "addc.u32 %4, 0, 0;"
        : "=r"(s[0]), "=r"(s[1]), "=r"(s[2]), "=r"(s[3]), "=r"(c), "=r"(t)
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]), "r"(b[2]), "r"(b[3]), "r"(cin));
    return c;
}

template <int N>
__device__ __forceinline__ void fe_cond_sub_p(uint32_t* r, const uint32_t* a, uint32_t carry, const uint32_t* p) {
    if constexpr (N == 8) cond_sub_chain8(r, a, carry, p);
    else if constexpr (N == 4) cond_sub_chain4(r, a, carry, p);
    else fe_cond_sub_p_portable<N>(r, a, carry, p);
}

// r = (a + b) mod p, inputs in [0, p)
template <int N>
__device__ __forceinline__ void fe_add(uint32_t* r, const uint32_t* a, const uint32_t* b, const uint32_t* p) {
    if constexpr (N == 8) {
        uint32_t s[8];
        uint32_t c = add_chain8(s, a, b);
        cond_sub_chain8(r, s, c, p);
    } else if constexpr (N == 4) {
        uint32_t s[4];
        uint32_t c = add_chain4(s, a, b);
        cond_sub_chain4(r, s, c, p);
    } else {
        fe_add_portable<N>(r, a, b, p);
    }
}

template <int N>
struct PtxChains;
template <>
struct PtxChains<8> {
    static __device__ __forceinline__ void mul_even(uint32_t* acc, const uint32_t* x, uint32_t y) { mul_pairs4(acc, x[0], x[2], x[4], x[6], y); }
    static __device__ __forceinline__ void mul_odd(uint32_t* acc, const uint32_t* x, uint32_t y) { mul_pairs4(acc, x[1], x[3], x[5], x[7], y); }
    static __device__ __forceinline__ uint32_t mad_even(uint32_t* acc, const uint32_t* x, uint32_t y, uint32_t cin = 0) { return mad_chain4(acc, x[0], x[2], x[4], x[6], y, cin); }
    static __device__ __forceinline__ uint32_t mad_odd(uint32_t* acc, const uint32_t* x, uint32_t y, uint32_t cin = 0) { return mad_chain4(acc, x[1], x[3], x[5], x[7], y, cin); }
    static __device__ __forceinline__ uint32_t mad_odd_fold(uint32_t& e0, uint32_t f0, uint32_t f1, uint32_t* acc, const uint32_t* x, uint32_t y) {
        return mad_chain4_fold(e0, f0, f1, acc, x[1], x[3], x[5], x[7], y);
    }
    static __device__ __forceinline__ uint32_t mad_odd_cbot(uint32_t* acc, const uint32_t* x, uint32_t y, uint32_t cbot) {
        return mad_chain4_cbot(acc, x[1], x[3], x[5], x[7], y, cbot);
    }
    static __device__ __forceinline__ uint32_t add(uint32_t* s, const uint32_t* a, const uint32_t* b) { return add_chain8(s, a, b); }
    static __device__ __forceinline__ uint32_t add_cin(uint32_t* s, const uint32_t* a, const uint32_t* b, uint32_t cin) { return add_chain8_cin(s, a, b, cin); }
};
template <>
struct PtxChains<4> {
    static __device__ __forceinline__ void mul_even(uint32_t* acc, const uint32_t* x, uint32_t y) { mul_pairs2(acc, x[0], x[2], y); }
    static __device__ __forceinline__ void mul_odd(uint32_t* acc, const uint32_t* x, uint32_t y) { mul_pairs2(acc, x[1], x[3], y); }
    static __device__ __forceinline__ uint32_t mad_even(uint32_t* acc, const uint32_t* x, uint32_t y, uint32_t cin = 0) { return mad_chain2(acc, x[0], x[2], y, cin); }
    static __device__ __forceinline__ uint32_t mad_odd(uint32_t* acc, const uint32_t* x, uint32_t y, uint32_t cin = 0) { return mad_chain2(acc, x[1], x[3], y, cin); }
    static __device__ __forceinline__ uint32_t mad_odd_fold(uint32_t& e0, uint32_t f0, uint32_t f1, uint32_t* acc, const uint32_t* x, uint32_t y) {
        return mad_chain2_fold(e0, f0, f1, acc, x[1], x[3], y);
    }
    static __device__ __forceinline__ uint32_t mad_odd_cbot(uint32_t* acc, const uint32_t* x, uint32_t y, uint32_t cbot) {
        return mad_chain2_cbot(acc, x[1], x[3], y, cbot);
    }
    static __device__ __forceinline__ uint32_t add(uint32_t* s, const uint32_t* a, const uint32_t* b) { return add_chain4(s, a, b); }
    static __device__ __forceinline__ uint32_t add_cin(uint32_t* s, const uint32_t* a, const uint32_t* b, uint32_t cin) { return add_chain4_cin(s, a, b, cin); }
};

template <int N>
__device__ __forceinline__ void fe_mont_mul_chain(uint32_t* r, const uint32_t* a, const uint32_t* b, const uint32_t* p, uint32_t n0inv) {
    using Ch = PtxChains<N>;
    uint32_t E[N], O[N];
    Ch::mul_even(E, a, b[0]);
    Ch::mul_odd(O, a, b[0]);
    uint32_t m = E[0] * n0inv;
    uint32_t cE = Ch::mad_even(E, p, m);
    uint32_t cO = Ch::mad_odd(O, p, m);
#pragma unroll
    for (int i = 1; i < N; i++) {
        // shift down one limb: new E = O (+ E[1] folded into limb 0), new O = E[2..] ++ (cE, cO)
        uint32_t nE[N], nO[N];
#pragma unroll
        for (int j = 1; j < N; j++) nE[j] = O[j];
#pragma unroll
        for (int j = 0; j < N - 2; j++) nO[j] = E[j + 2];
        nO[N - 2] = cE;
        nO[N - 1] = cO;
        cO = Ch::mad_odd_fold(nE[0], O[0], E[1], nO, a, b[i]);   // nE[0] = O[0] + E[1]; carry rides into the odd chain
        cE = Ch::mad_even(nE, a, b[i]);
        m = nE[0] * n0inv;
        cE = Ch::mad_even(nE, p, m, cE);
        cO = Ch::mad_odd(nO, p, m, cO);
#pragma unroll
        for (int j = 0; j < N; j++) {
            E[j] = nE[j];
            O[j] = nO[j];
        }
    }
    // final shift + merge of the two accumulators: limb j = E[j+1] + O[j], limb N-1 = cE + O[N-1], top = cO
    uint32_t t[N], up[N];
#pragma unroll
    for (int j = 0; j < N - 1; j++) up[j] = E[j + 1];
    up[N - 1] = cE;
    uint32_t top;
    if constexpr (N == 8) top = add_chain8(t, up, O) + cO;
    else top = add_chain4(t, up, O) + cO;
    fe_cond_sub_p<N>(r, t, top, p);
}

// fe_mont_mul_chain<8> for a modulus whose low 64 bits are 2^64 - 2^32 + 1 (p0 = 1, p1 = 2^32 - 1: BLS12-381 Fr), so that
// n0inv = 2^32 - 1.  A row's multiplier is m = -T0 mod 2^32 (no multiply), p0 * m = m and p1 * m = (m - [m != 0] : T0): the
// reduction of a row takes 6 wide products instead of 8, a product 112 multiplies instead of 136.  Every chain adds the
// same integers as in fe_mont_mul_chain<8>, so T + m p, the carries and the result are bit for bit the same for every input
// that product accepts (a b < p R).
__device__ __forceinline__ void fe_mont_mul_low64(uint32_t* r, const uint32_t* a, const uint32_t* b, const uint32_t* p) {
    using Ch = PtxChains<8>;
    uint32_t E[8], O[8], m, mh;
    Ch::mul_even(E, a, b[0]);
    Ch::mul_odd(O, a, b[0]);
    low64_m(m, mh, E[0]);
    uint32_t cO = mad_chain4_low_odd(O, E[0], mh, p[3], p[5], p[7], m, 0);
    uint32_t cE = mad_chain4_low_even(E, p[2], p[4], p[6], m, 0);
#pragma unroll
    for (int i = 1; i < 8; i++) {
        uint32_t nE[8], nO[8];
#pragma unroll
        for (int j = 1; j < 8; j++) nE[j] = O[j];
#pragma unroll
        for (int j = 0; j < 6; j++) nO[j] = E[j + 2];
        nO[6] = cE;
        nO[7] = cO;
        cO = Ch::mad_odd_fold(nE[0], O[0], E[1], nO, a, b[i]);
        cE = Ch::mad_even(nE, a, b[i]);
        low64_m(m, mh, nE[0]);
        cO = mad_chain4_low_odd(nO, nE[0], mh, p[3], p[5], p[7], m, cO);
        cE = mad_chain4_low_even(nE, p[2], p[4], p[6], m, cE);
#pragma unroll
        for (int j = 0; j < 8; j++) {
            E[j] = nE[j];
            O[j] = nO[j];
        }
    }
    uint32_t t[8], up[8];
#pragma unroll
    for (int j = 0; j < 7; j++) up[j] = E[j + 1];
    up[7] = cE;
    const uint32_t top = add_chain8(t, up, O) + cO;
    cond_sub_chain8(r, t, top, p);
}

// ---- lazy reduction (the R1CS check: one Montgomery reduction per linear combination instead of one per term) --------
// A linear combination sum_k coef_k * z_k of Montgomery residues is accumulated as the plain integer
//     T = sum_k (z_k R)(coef_k R)  +  sum over coefficient-one terms of (z_k R) * R            (R = 2^(32N)),
// 2N + 1 limbs (every term is below p R < R^2: the top limb counts the overflows), and reduced ONCE: REDC(T) = T / R mod p
// = R sum_k coef_k z_k.  A term costs the N^2 multiplications of the plain product instead of the 2 N^2 of a Montgomery
// product, a linear combination N^2 more for its reduction.

// P (2N limbs) = a * b as plain integers: the rows of fe_mont_mul_chain without the reduction steps
template <int N>
__device__ __forceinline__ void fe_mul_wide(uint32_t* P, const uint32_t* a, const uint32_t* b) {
    using Ch = PtxChains<N>;
    uint32_t E[N], O[N];
    Ch::mul_even(E, a, b[0]);
    Ch::mul_odd(O, a, b[0]);
    P[0] = E[0];
    uint32_t cE = 0, cO = 0;
#pragma unroll
    for (int i = 1; i < N; i++) {
        uint32_t nE[N], nO[N];
#pragma unroll
        for (int j = 1; j < N; j++) nE[j] = O[j];
#pragma unroll
        for (int j = 0; j < N - 2; j++) nO[j] = E[j + 2];
        nO[N - 2] = cE;
        nO[N - 1] = cO;
        cO = Ch::mad_odd_fold(nE[0], O[0], E[1], nO, a, b[i]);
        cE = Ch::mad_even(nE, a, b[i]);
        P[i] = nE[0];  // nothing lands on this limb any more
#pragma unroll
        for (int j = 0; j < N; j++) {
            E[j] = nE[j];
            O[j] = nO[j];
        }
    }
    uint32_t up[N];
#pragma unroll
    for (int j = 0; j < N - 1; j++) up[j] = E[j + 1];
    up[N - 1] = cE;
    Ch::add(P + N, up, O);  // the product is below R^2: no carry out, cO = 0
}

// r = (a + m p) / R for the N-limb integer a (m chosen limb by limb so that the division is exact): a value in [0, p],
// congruent to a / R.  NOT reduced below p: the caller adds the upper half of its accumulator and reduces once.
template <int N>
__device__ __forceinline__ void fe_redc_low(uint32_t* r, const uint32_t* a, const uint32_t* p, uint32_t n0inv) {
    using Ch = PtxChains<N>;
    uint32_t E[N], O[N];
#pragma unroll
    for (int j = 0; j < N; j += 2) {  // a as the first row of a product by 1: even limbs in E, odd limbs in O
        E[j] = a[j];
        E[j + 1] = 0;
        O[j] = a[j + 1];
        O[j + 1] = 0;
    }
    uint32_t m = E[0] * n0inv;
    uint32_t cE = Ch::mad_even(E, p, m);
    uint32_t cO = Ch::mad_odd(O, p, m);
#pragma unroll
    for (int i = 1; i < N; i++) {
        uint32_t nE[N], nO[N];
#pragma unroll
        for (int j = 1; j < N; j++) nE[j] = O[j];
#pragma unroll
        for (int j = 0; j < N - 2; j++) nO[j] = E[j + 2];
        nO[N - 2] = cE;
        nO[N - 1] = cO;
        uint32_t cf;
        asm("add.cc.u32 %0, %2, %3;\n\t"
            "addc.u32 %1, 0, 0;"
            : "=r"(nE[0]), "=r"(cf)
            : "r"(O[0]), "r"(E[1]));
        m = nE[0] * n0inv;
        cE = Ch::mad_even(nE, p, m);
        cO = Ch::mad_odd_cbot(nO, p, m, cf);
#pragma unroll
        for (int j = 0; j < N; j++) {
            E[j] = nE[j];
            O[j] = nO[j];
        }
    }
    uint32_t up[N];
#pragma unroll
    for (int j = 0; j < N - 1; j++) up[j] = E[j + 1];
    up[N - 1] = cE;
    Ch::add(r, up, O);  // <= p < R: no carry out
}

// T (2N + 1 limbs) += a * b
template <int N>
__device__ __forceinline__ void fe_lazy_mad(uint32_t* T, const uint32_t* a, const uint32_t* b) {
    using Ch = PtxChains<N>;
    uint32_t P[2 * N];
    fe_mul_wide<N>(P, a, b);
    const uint32_t c = Ch::add(T, T, P);
    T[2 * N] += Ch::add_cin(T + N, T + N, P + N, c);
}
// T += a * R  (a term with coefficient one)
template <int N>
__device__ __forceinline__ void fe_lazy_add_one(uint32_t* T, const uint32_t* a) {
    using Ch = PtxChains<N>;
    T[2 * N] += Ch::add(T + N, T + N, a);
}
// r = T / R mod p, fully reduced.  T < (k + 1) p R after k terms, so the quotient by p is small: subtract p while it fits.
// `low_half`: false when only coefficient-one terms were added (the lower N limbs are zero: the division by R is a shift).
template <int N>
__device__ __forceinline__ void fe_lazy_finish(uint32_t* r, const uint32_t* T, const uint32_t* p, uint32_t n0inv, bool low_half = true) {
    using Ch = PtxChains<N>;
    uint32_t s[N];
    uint32_t top = T[2 * N];
    if (low_half) {
        uint32_t lo[N];
        fe_redc_low<N>(lo, T, p, n0inv);
        top += Ch::add(s, lo, T + N);
    } else {
#pragma unroll
        for (int j = 0; j < N; j++) s[j] = T[N + j];
    }
    for (;;) {
        uint32_t d[N];
        uint32_t borrow = 0;
#pragma unroll
        for (int j = 0; j < N; j++) {  // d = s - p limb by limb (compiles to one borrow chain)
            const uint64_t x = (uint64_t)s[j] - p[j] - borrow;
            d[j] = (uint32_t)x;
            borrow = (uint32_t)(x >> 63);
        }
        if (top == 0 && borrow) break;  // (top : s) < p
        top -= borrow;
#pragma unroll
        for (int j = 0; j < N; j++) s[j] = d[j];
    }
#pragma unroll
    for (int j = 0; j < N; j++) r[j] = s[j];
}

// Two-limb fields (33..64-bit moduli) as ONE 64-bit limb: the 128-bit product is mul.lo.u64 / mul.hi.u64, the Montgomery
// step one more product pair - or, for the Goldilocks prime p = 2^64 - 2^32 + 1, no product at all: p^-1 = 1 + 2^32
// (mod 2^64), so m = lo + (lo << 32) and m * p / 2^64 = m - (m >> 32) - [the add overflowed], all shifts and adds.
// Same contract as the CIOS form: a * b < p * 2^64, result fully reduced.  -p^-1 mod 2^64 is rebuilt from its low half
// (n0inv) by one Newton step; the compiler hoists that out of the gate loop (it depends on the field only).
__device__ __forceinline__ void fe_mont_mul_u64(uint32_t* r, const uint32_t* a, const uint32_t* b, const uint32_t* p, uint32_t n0inv) {
    const uint64_t A = (uint64_t)a[1] << 32 | a[0], B = (uint64_t)b[1] << 32 | b[0], P = (uint64_t)p[1] << 32 | p[0];
    const uint64_t lo = A * B, hi = __umul64hi(A, B);
    uint64_t res;
    if (P == 0xFFFFFFFF00000001ull) {
        const uint64_t m = lo + (lo << 32);
        const uint64_t e = m < lo ? 1u : 0u;
        const uint64_t q = m - (m >> 32) - e;     // m * p / 2^64
        res = hi - q;
        if (hi < q) res -= 0xFFFFFFFFull;         // + p (mod 2^64)
        if (res >= P) res -= P;
    } else {
        uint64_t ninv = (uint64_t)n0inv;                 // -p^-1 mod 2^32
        ninv = 0 - ninv;                                 // p^-1 mod 2^32 (as a 64-bit value: correct in the low half)
        ninv *= 2 - P * ninv;                            // Newton: p^-1 mod 2^64
        const uint64_t m = lo * (0 - ninv);
        const uint64_t uh = __umul64hi(m, P);            // lo + low(m * P) = 0 mod 2^64: carries exactly when lo != 0
        res = hi + uh;
        uint64_t carry = res < hi ? 1u : 0u;
        const uint64_t c0 = lo != 0 ? 1u : 0u;
        res += c0;
        carry |= res < c0 ? 1u : 0u;
        if (carry || res >= P) res -= P;
    }
    r[0] = (uint32_t)res;
    r[1] = (uint32_t)(res >> 32);
}

template <int N>
__device__ __forceinline__ void fe_mont_mul(uint32_t* r, const uint32_t* a, const uint32_t* b, const uint32_t* p, uint32_t n0inv) {
    if constexpr (N == 8 || N == 4) fe_mont_mul_chain<N>(r, a, b, p, n0inv);
#ifndef ZKB_NO_U64_FIELD
    else if constexpr (N == 2) fe_mont_mul_u64(r, a, b, p, n0inv);
#endif
    else fe_mont_mul_portable<N>(r, a, b, p, n0inv);
}

// the hot kernels' product: FORM is the modulus's FieldParams::mul_form, a template parameter chosen at launch (a branch on
// it inside the kernel would hold both products' registers)
template <int N, uint32_t FORM>
__device__ __forceinline__ void fe_mont_mul_form(uint32_t* r, const uint32_t* a, const uint32_t* b, const uint32_t* p, uint32_t n0inv) {
    if constexpr (N == 8 && FORM == kMulFormLow64) fe_mont_mul_low64(r, a, b, p);
    else fe_mont_mul<N>(r, a, b, p, n0inv);
}

}  // namespace zkb
#endif
