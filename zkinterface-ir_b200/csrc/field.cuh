// Multi-limb prime-field arithmetic shared by host and device.
//
// Replaces the arbitrary-precision `(a op b) % m` of the reference's
// PlaintextBackend (rust/src/consumers/evaluator.rs:908-922) by fixed-width
// Montgomery arithmetic on N little-endian 32-bit limbs (N = 1, 2, 4, 8:
// p < 2^32, 2^64, 2^128, 2^256).  Values are always kept fully reduced in
// [0, p), in Montgomery form x*R mod p with R = 2^(32N), so "== 0" on the
// stored limbs is exactly the reference's `is_zero()` on a reduced value.
//
// Everything here is __host__ __device__ so the same code is unit-tested on the
// CPU (tests/native/field_host_test.cpp) and runs inside the sm_100a kernels.
// The device build swaps fe_mont_mul for a PTX mad.lo.cc/madc.hi.cc carry-chain
// version (field_ptx.cuh); the portable one below is its in-kernel cross-check.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define ZKB_HD __host__ __device__ __forceinline__
#else
#define ZKB_HD inline
#endif

namespace zkb {

constexpr int kMaxLimbs = 8;

// Field description, passed to kernels by value (lives in the constant bank).
struct FieldParams {
    uint32_t p[kMaxLimbs];     // modulus
    uint32_t r2[kMaxLimbs];    // R^2 mod p   (to Montgomery form)
    uint32_t one[kMaxLimbs];   // R mod p     (Montgomery 1)
    uint32_t n0inv;            // -p^{-1} mod 2^32
    uint32_t nlimb;            // 1, 2, 4 or 8
    uint32_t top_mask;         // mask of the bits of limb N-1 that can be set in a value < 2^bitlen(p)
    uint32_t mul_form;         // kMulForm*: which Montgomery product the hot kernels may run for this modulus
};

// FieldParams::mul_form (Program::set_field)
enum : uint32_t {
    kMulFormGeneric = 0,  // any odd p
    kMulFormLow64 = 1,    // 8 limbs and p = 2^64 - 2^32 + 1 mod 2^64 (BLS12-381 Fr): field_ptx.cuh fe_mont_mul_low64
};

template <int N>
ZKB_HD bool fe_is_zero(const uint32_t* a) {
    uint32_t acc = 0;
#pragma unroll
    for (int i = 0; i < N; i++) acc |= a[i];
    return acc == 0;
}

// r = a - p if (carry || a >= p) else a.   a has an extra carry bit `carry`.
template <int N>
ZKB_HD void fe_cond_sub_p_portable(uint32_t* r, const uint32_t* a, uint32_t carry, const uint32_t* p) {
    uint32_t d[N];
    uint32_t borrow = 0;
#pragma unroll
    for (int i = 0; i < N; i++) {
        uint64_t t = (uint64_t)a[i] - p[i] - borrow;
        d[i] = (uint32_t)t;
        borrow = (uint32_t)(t >> 63);
    }
    bool use_d = (carry != 0) || (borrow == 0);
#pragma unroll
    for (int i = 0; i < N; i++) r[i] = use_d ? d[i] : a[i];
}

// r = (a + b) mod p, inputs in [0, p)
template <int N>
ZKB_HD void fe_add_portable(uint32_t* r, const uint32_t* a, const uint32_t* b, const uint32_t* p) {
    uint32_t s[N];
    uint64_t c = 0;
#pragma unroll
    for (int i = 0; i < N; i++) {
        c += (uint64_t)a[i] + b[i];
        s[i] = (uint32_t)c;
        c >>= 32;
    }
    fe_cond_sub_p_portable<N>(r, s, (uint32_t)c, p);
}

// Montgomery product r = a*b/R mod p (CIOS).  a*b < p*R is enough (so one operand
// may be any N-limb integer when the other is < p); result fully reduced.
template <int N>
ZKB_HD void fe_mont_mul_portable(uint32_t* r, const uint32_t* a, const uint32_t* b, const uint32_t* p,
                                 uint32_t n0inv) {
    uint32_t t[N + 2];
#pragma unroll
    for (int i = 0; i < N + 2; i++) t[i] = 0;
#pragma unroll
    for (int i = 0; i < N; i++) {
        uint64_t c = 0;
#pragma unroll
        for (int j = 0; j < N; j++) {
            c += (uint64_t)a[j] * b[i] + t[j];
            t[j] = (uint32_t)c;
            c >>= 32;
        }
        c += t[N];
        t[N] = (uint32_t)c;
        t[N + 1] = (uint32_t)(c >> 32);
        uint32_t m = t[0] * n0inv;
        c = (uint64_t)m * p[0] + t[0];
        c >>= 32;
#pragma unroll
        for (int j = 1; j < N; j++) {
            c += (uint64_t)m * p[j] + t[j];
            t[j - 1] = (uint32_t)c;
            c >>= 32;
        }
        c += t[N];
        t[N - 1] = (uint32_t)c;
        t[N] = t[N + 1] + (uint32_t)(c >> 32);
    }
    fe_cond_sub_p_portable<N>(r, t, t[N], p);
}

// the device pass gets fe_mont_mul / fe_add / fe_cond_sub_p from field_ptx.cuh (PTX carry chains); host code and
// -DZKB_NO_PTX_FIELD use the portable ones
#if !(defined(__CUDA_ARCH__) && !defined(ZKB_NO_PTX_FIELD))
template <int N>
ZKB_HD void fe_mont_mul(uint32_t* r, const uint32_t* a, const uint32_t* b, const uint32_t* p, uint32_t n0inv) {
    fe_mont_mul_portable<N>(r, a, b, p, n0inv);
}
template <int N, uint32_t FORM>
ZKB_HD void fe_mont_mul_form(uint32_t* r, const uint32_t* a, const uint32_t* b, const uint32_t* p, uint32_t n0inv) {
    fe_mont_mul_portable<N>(r, a, b, p, n0inv);
}
template <int N>
ZKB_HD void fe_add(uint32_t* r, const uint32_t* a, const uint32_t* b, const uint32_t* p) {
    fe_add_portable<N>(r, a, b, p);
}
template <int N>
ZKB_HD void fe_cond_sub_p(uint32_t* r, const uint32_t* a, uint32_t carry, const uint32_t* p) {
    fe_cond_sub_p_portable<N>(r, a, carry, p);
}
// lazy reduction (see field_ptx.cuh): T is a plain integer of 2N + 1 limbs
template <int N>
ZKB_HD void fe_mul_wide(uint32_t* P, const uint32_t* a, const uint32_t* b) {
    for (int k = 0; k < 2 * N; k++) P[k] = 0;
    for (int i = 0; i < N; i++) {
        uint64_t carry = 0;
        for (int j = 0; j < N; j++) {
            const uint64_t t = (uint64_t)P[i + j] + (uint64_t)a[j] * b[i] + carry;
            P[i + j] = (uint32_t)t;
            carry = t >> 32;
        }
        P[i + N] = (uint32_t)carry;
    }
}
template <int N>
ZKB_HD void fe_lazy_mad(uint32_t* T, const uint32_t* a, const uint32_t* b) {
    for (int i = 0; i < N; i++) {
        uint64_t carry = 0;
        for (int j = 0; j < N; j++) {
            const uint64_t t = (uint64_t)T[i + j] + (uint64_t)a[j] * b[i] + carry;
            T[i + j] = (uint32_t)t;
            carry = t >> 32;
        }
        for (int k = i + N; k <= 2 * N && carry; k++) {
            const uint64_t t = (uint64_t)T[k] + carry;
            T[k] = (uint32_t)t;
            carry = t >> 32;
        }
    }
}
template <int N>
ZKB_HD void fe_lazy_add_one(uint32_t* T, const uint32_t* a) {
    uint64_t carry = 0;
    for (int j = 0; j < N; j++) {
        const uint64_t t = (uint64_t)T[N + j] + a[j] + carry;
        T[N + j] = (uint32_t)t;
        carry = t >> 32;
    }
    T[2 * N] += (uint32_t)carry;
}
template <int N>
ZKB_HD void fe_lazy_finish(uint32_t* r, const uint32_t* T, const uint32_t* p, uint32_t n0inv, bool low_half = true) {
    uint32_t t[2 * N + 2];
    for (int k = 0; k <= 2 * N; k++) t[k] = T[k];
    t[2 * N + 1] = 0;
    if (low_half)
        for (int i = 0; i < N; i++) {
            const uint32_t m = t[i] * n0inv;
            uint64_t carry = 0;
            for (int j = 0; j < N; j++) {
                const uint64_t x = (uint64_t)t[i + j] + (uint64_t)m * p[j] + carry;
                t[i + j] = (uint32_t)x;
                carry = x >> 32;
            }
            for (int k = i + N; k <= 2 * N + 1 && carry; k++) {
                const uint64_t x = (uint64_t)t[k] + carry;
                t[k] = (uint32_t)x;
                carry = x >> 32;
            }
        }
    uint32_t s[N], top = t[2 * N];
    for (int j = 0; j < N; j++) s[j] = t[N + j];
    for (;;) {
        uint32_t d[N], borrow = 0;
        for (int j = 0; j < N; j++) {
            const uint64_t x = (uint64_t)s[j] - p[j] - borrow;
            d[j] = (uint32_t)x;
            borrow = (uint32_t)(x >> 63);
        }
        if (top == 0 && borrow) break;
        top -= borrow;
        for (int j = 0; j < N; j++) s[j] = d[j];
    }
    for (int j = 0; j < N; j++) r[j] = s[j];
}
#else
template <int N>
__device__ __forceinline__ void fe_cond_sub_p(uint32_t* r, const uint32_t* a, uint32_t carry, const uint32_t* p);
#endif

// Bitwise gates on canonical (non-Montgomery) residues, as PlaintextBackend::and / ::xor
// (evaluator.rs:924-930): (a & b) % m and (a ^ b) % m for a, b < p.  a & b <= a < p needs no
// reduction; a ^ b < 2^bitlen(p) <= 2p needs at most one subtraction.
template <int N>
ZKB_HD void fe_and_canon(uint32_t* r, const uint32_t* a, const uint32_t* b) {
#pragma unroll
    for (int i = 0; i < N; i++) r[i] = a[i] & b[i];
}
template <int N>
ZKB_HD void fe_xor_canon(uint32_t* r, const uint32_t* a, const uint32_t* b, const uint32_t* p) {
    uint32_t x[N];
#pragma unroll
    for (int i = 0; i < N; i++) x[i] = a[i] ^ b[i];
    fe_cond_sub_p<N>(r, x, 0, p);
}

}  // namespace zkb
