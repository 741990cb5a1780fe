// Goldilocks (p = 2^64 - 2^32 + 1) and GoldilocksExt2 = F[X]/(X^2 - 7) arithmetic, host + device.
//
// Replaces the `goldilocks` crate the reference links (/root/reference/Cargo.toml:28,67-68; used at
// /root/reference/bfv-gkr/src/sk_encryption_circuit.rs:539). Elements are canonical u64 (< p) in memory; the
// reduction is the 64x64->128 mul.lo/mul.hi + "2^64 = 2^32 - 1, 2^96 = -1" fold (IMAD pipe, no tensor cores).
#pragma once
#include <cstdint>

#if defined(__CUDACC__)
#define HG_HD __host__ __device__ __forceinline__
#else
#define HG_HD inline
#endif

namespace hg {

typedef uint64_t u64;
typedef uint32_t u32;

constexpr u64 GL_P = 0xFFFFFFFF00000001ULL;
constexpr u64 GL_EPS = 0xFFFFFFFFULL;  // 2^64 mod p

// On the host (transcript serialisation: ~18 000 extension products per proof) the wrap tests of random field elements are
// coin flips for the branch predictor, so the host versions are written without data-dependent branches: 43 -> 12 ns per
// extension multiply-add, 0.8 -> 0.4 ms of serialisation per proof. The device code is unchanged.
HG_HD u64 gl_add(u64 a, u64 b) {
    u64 s = a + b;
#if defined(__CUDA_ARCH__)
    if (s < a) s += GL_EPS;       // wrapped: + 2^64 = + EPS. a, b < p gives s = a + b - 2^64 <= p - 2 - EPS, so s + EPS < p
    else if (s >= GL_P) s -= GL_P;
#else
    s += (0 - (u64)(s < a)) & GL_EPS;   // after a wrap the sum is < p - EPS, so at most one of the two corrections applies
    s -= (0 - (u64)(s >= GL_P)) & GL_P;
#endif
    return s;
}
HG_HD u64 gl_sub(u64 a, u64 b) {
    u64 d = a - b;
#if defined(__CUDA_ARCH__)
    if (a < b) d -= GL_EPS;       // wrapped: - 2^64 = - EPS
#else
    d -= (0 - (u64)(a < b)) & GL_EPS;
#endif
    return d;
}
HG_HD u64 gl_neg(u64 a) { return a ? GL_P - a : 0; }
HG_HD u64 gl_dbl(u64 a) { return gl_add(a, a); }

HG_HD void mul_wide(u64 a, u64 b, u64& lo, u64& hi) {
#if defined(__CUDA_ARCH__)
    lo = a * b;
    hi = __umul64hi(a, b);
#else
    unsigned __int128 p = (unsigned __int128)a * b;
    lo = (u64)p;
    hi = (u64)(p >> 64);
#endif
}
// (lo + 2^64 hi) mod p, canonical
HG_HD u64 gl_reduce128(u64 lo, u64 hi) {
    u64 hi_hi = hi >> 32, hi_lo = hi & GL_EPS;
    u64 t0 = lo - hi_hi;
    u64 t1 = (hi_lo << 32) - hi_lo;  // hi_lo * (2^32 - 1)
#if defined(__CUDA_ARCH__)
    if (lo < hi_hi) t0 -= GL_EPS;
    u64 r = t0 + t1;
    if (r < t1) r += GL_EPS;
    if (r >= GL_P) r -= GL_P;
#else
    t0 -= (0 - (u64)(lo < hi_hi)) & GL_EPS;
    u64 r = t0 + t1;
    r += (0 - (u64)(r < t1)) & GL_EPS;
    r -= (0 - (u64)(r >= GL_P)) & GL_P;
#endif
    return r;
}
HG_HD u64 gl_mul(u64 a, u64 b) {
    u64 lo, hi;
    mul_wide(a, b, lo, hi);
    return gl_reduce128(lo, hi);
}
HG_HD u64 gl_from_u64(u64 x) { return x >= GL_P ? x - GL_P : x; }
HG_HD u64 gl_pow(u64 b, u64 e) {
    u64 r = 1;
    while (e) { if (e & 1) r = gl_mul(r, b); b = gl_mul(b, b); e >>= 1; }
    return r;
}
HG_HD u64 gl_inv(u64 a) { return gl_pow(a, GL_P - 2); }

// ------------------------------------------------------------------ Ext2
struct __align__(16) gl2 {
    u64 c0, c1;
};
HG_HD gl2 gl2_make(u64 a, u64 b) { gl2 r; r.c0 = a; r.c1 = b; return r; }
HG_HD gl2 gl2_zero() { return gl2_make(0, 0); }
HG_HD gl2 gl2_one() { return gl2_make(1, 0); }
HG_HD gl2 gl2_lift(u64 a) { return gl2_make(a, 0); }
HG_HD gl2 gl2_add(gl2 a, gl2 b) { return gl2_make(gl_add(a.c0, b.c0), gl_add(a.c1, b.c1)); }
HG_HD gl2 gl2_sub(gl2 a, gl2 b) { return gl2_make(gl_sub(a.c0, b.c0), gl_sub(a.c1, b.c1)); }
HG_HD gl2 gl2_neg(gl2 a) { return gl2_make(gl_neg(a.c0), gl_neg(a.c1)); }
HG_HD u64 gl_mul7(u64 a) {  // 7a = 8a - a
    u64 lo = a << 3, hi = a >> 61;
    u64 r = gl_reduce128(lo, hi);
    return gl_sub(r, a);
}
HG_HD gl2 gl2_mul(gl2 a, gl2 b) {
#if !defined(__CUDA_ARCH__)
    {   // host: four 64x64 products, three reductions. c0 = a0 b0 + 7 (a1 b1 mod p): (p-1)^2 + 7 (p-1) < 2^128;
        // c1 = a0 b1 + a1 b0 with the carry out of 128 bits folded in as 2^128 = -2^32 (mod p)
        typedef unsigned __int128 u128;
        const u128 p11 = (u128)a.c1 * b.c1;
        const u64 v11 = gl_reduce128((u64)p11, (u64)(p11 >> 64));
        const u128 t = (u128)a.c0 * b.c0 + (u128)v11 * 7;
        const u128 p01 = (u128)a.c0 * b.c1, s1 = p01 + (u128)a.c1 * b.c0;
        const u64 carry = (u64)(s1 < p01);
        return gl2_make(gl_reduce128((u64)t, (u64)(t >> 64)), gl_sub(gl_reduce128((u64)s1, (u64)(s1 >> 64)), carry << 32));
    }
#endif
    // Karatsuba: c0 = a0 b0 + 7 a1 b1, c1 = (a0 + a1)(b0 + b1) - a0 b0 - a1 b1
    u64 v0 = gl_mul(a.c0, b.c0), v1 = gl_mul(a.c1, b.c1);
    u64 m = gl_mul(gl_add(a.c0, a.c1), gl_add(b.c0, b.c1));
    return gl2_make(gl_add(v0, gl_mul7(v1)), gl_sub(gl_sub(m, v0), v1));
}
HG_HD gl2 gl2_mul_base(gl2 a, u64 b) { return gl2_make(gl_mul(a.c0, b), gl_mul(a.c1, b)); }
HG_HD gl2 gl2_dbl(gl2 a) { return gl2_add(a, a); }
HG_HD bool gl2_eq(gl2 a, gl2 b) { return a.c0 == b.c0 && a.c1 == b.c1; }
HG_HD gl2 gl2_inv(gl2 a) {
    u64 n = gl_sub(gl_mul(a.c0, a.c0), gl_mul7(gl_mul(a.c1, a.c1)));
    u64 ni = gl_inv(n);
    return gl2_make(gl_mul(a.c0, ni), gl_mul(gl_neg(a.c1), ni));
}


// ------------------------------------------------------------------ device fast path: carry chains + lazy accumulation
// The generic functions above compile to long compare/select sequences that saturate the ALU pipe (profiles/ round 1).
// The hot kernels use these instead:
//   * table elements in memory are always CANONICAL (< p);
//   * products are accumulated UNREDUCED in a 160-bit accumulator (lo, hi, carry word) and reduced once;
//   * subtraction needs only its subtrahend canonical; results are "lazy" (any representative in [0, 2^64)).
// Contracts, per primitive ("lazy" = any u64, "canonical" = < p). tests/test_field_probe.py checks each one at its limit.
//   acc_mad(a, x, y), acc_add(a, x)   x, y lazy. acc_mad adds at most 1 to e4 and at most 2 to o2, acc_add at most 1 to e4.
//   acc_reduce                        exact and canonical for any e01, e23, o01, o2 and e4 <= 2^32 - 3. From acc_zero / acc_from
//                                     that is n acc_mad and m acc_add with 2n <= 2^32 - 1 and n + m <= 2^32 - 3: 2^31 - 1 products.
//   xacc_mad, xacc_mad_base           x, y lazy. xacc_mad adds one product to a00 and a11 and two to ax, xacc_mad_base one to
//                                     a00 and ax. xacc_reduce adds one more product to (a copy of) a00, which must have room
//                                     for it. Output canonical.
//   gl_sub_cs(a, b)                   b canonical, a lazy; output lazy, canonical when a is.
//   gl_add_cs(a, b)                   a canonical, b lazy; output lazy (may be p, a non-canonical zero).
//   gl_canon(r)                       r lazy; output canonical.
//   gl_mul_fast, gl2_mul_fast, GlField::fmul_any   operands lazy; output canonical.
//   gl2_fold, GlField::fold_scaled    canonical in (a0, a1, r, c, cr and fold_aux's r7), canonical out.
//   GlField::slope                    canonical in; output canonical. at_m1, q_at_m1: canonical in, lazy out.
#if defined(__CUDACC__)
// Unreduced sum of 64x64-bit products, kept as TWO column accumulators so that every 32x32 partial product lands on an
// aligned 64-bit register pair and one IMAD.WIDE.U32 (with carry) adds it:
//     value = (e01 + 2^64 e23 + 2^128 e4)  +  2^32 (o01 + 2^64 o2)
// "even" columns take x0*y0 (weight 2^0) and x1*y1 (2^64), "odd" columns the cross products (2^32). acc_mad is
// 4 IMAD.WIDE.U32 + 3 carry adds (the single-accumulator form needed 15 instructions); the columns are merged once, in
// acc_reduce. Capacity: 2^31 - 1 products (o2 takes up to 2 carries per product), e4 <= 2^32 - 3 at acc_reduce.
struct acc192 {
    u64 e01, e23, o01;
    u32 e4, o2;
};
__device__ __forceinline__ acc192 acc_zero() { acc192 a; a.e01 = 0; a.e23 = 0; a.o01 = 0; a.e4 = 0; a.o2 = 0; return a; }
__device__ __forceinline__ acc192 acc_from(u64 v) { acc192 a = acc_zero(); a.e01 = v; return a; }
// a += x * y   (x, y any 64-bit values)
__device__ __forceinline__ void acc_mad(acc192& a, u64 x, u64 y) {
    asm("{\n\t.reg .u32 x0, x1, y0, y1, a0, a1, a2, a3, b0, b1;\n\t"
        "mov.b64 {x0, x1}, %5;\n\tmov.b64 {y0, y1}, %6;\n\t"
        "mov.b64 {a0, a1}, %0;\n\tmov.b64 {a2, a3}, %1;\n\tmov.b64 {b0, b1}, %3;\n\t"
        "mad.lo.cc.u32 a0, x0, y0, a0;\n\t"
        "madc.hi.cc.u32 a1, x0, y0, a1;\n\t"
        "madc.lo.cc.u32 a2, x1, y1, a2;\n\t"
        "madc.hi.cc.u32 a3, x1, y1, a3;\n\t"
        "addc.u32 %2, %2, 0;\n\t"
        "mad.lo.cc.u32 b0, x0, y1, b0;\n\t"
        "madc.hi.cc.u32 b1, x0, y1, b1;\n\t"
        "addc.u32 %4, %4, 0;\n\t"
        "mad.lo.cc.u32 b0, x1, y0, b0;\n\t"
        "madc.hi.cc.u32 b1, x1, y0, b1;\n\t"
        "addc.u32 %4, %4, 0;\n\t"
        "mov.b64 %0, {a0, a1};\n\tmov.b64 %1, {a2, a3};\n\tmov.b64 %3, {b0, b1};\n\t}"
        : "+l"(a.e01), "+l"(a.e23), "+r"(a.e4), "+l"(a.o01), "+r"(a.o2)
        : "l"(x), "l"(y));
}
__device__ __forceinline__ void acc_add(acc192& a, u64 x) {
    asm("add.cc.u64 %0, %0, %3; addc.cc.u64 %1, %1, 0; addc.u32 %2, %2, 0;" : "+l"(a.e01), "+l"(a.e23), "+r"(a.e4) : "l"(x));
}
__device__ __forceinline__ void acc_merge(acc192& a, const acc192& b) {
    asm("add.cc.u64 %0, %0, %3; addc.cc.u64 %1, %1, %4; addc.u32 %2, %2, %5;" : "+l"(a.e01), "+l"(a.e23), "+r"(a.e4) : "l"(b.e01), "l"(b.e23), "r"(b.e4));
    asm("add.cc.u64 %0, %0, %2; addc.u32 %1, %1, %3;" : "+l"(a.o01), "+r"(a.o2) : "l"(b.o01), "r"(b.o2));
}
// a - b mod p for CANONICAL b (a may be lazy); result lazy, canonical when a is canonical
__device__ __forceinline__ u64 gl_sub_cs(u64 a, u64 b) {
    u64 d;
    u32 m;
    asm("sub.cc.u64 %0, %2, %3; subc.u32 %1, 0, 0;" : "=l"(d), "=r"(m) : "l"(a), "l"(b));
    return d - (u64)m;  // m = 0xFFFFFFFF = EPS on borrow
}
// a + b mod p for CANONICAL a (b may be lazy); result lazy
__device__ __forceinline__ u64 gl_add_cs(u64 a, u64 b) {
    u64 s;
    u32 c;
    asm("add.cc.u64 %0, %2, %3; addc.u32 %1, 0, 0;" : "=l"(s), "=r"(c) : "l"(a), "l"(b));
    return s + (u64)(0u - c);  // + EPS on carry; cannot wrap twice because a < p
}
// lazy -> canonical
__device__ __forceinline__ u64 gl_canon(u64 r) {
    u64 t;
    u32 c;
    asm("add.cc.u64 %0, %2, %3; addc.u32 %1, 0, 0;" : "=l"(t), "=r"(c) : "l"(r), "l"(GL_EPS));  // t = r - p (mod 2^64), carry iff r >= p
    return c ? t : r;
}
// value mod p, canonical.  2^64 = 2^32 - 1, 2^96 = -1, 2^128 = -2^32 (mod p)
__device__ __forceinline__ u64 acc_reduce(const acc192& a) {
    // merge the odd columns: (lo, hi, c) = E + 2^32 O. (e1, e2, e3) + (o0, o1, o2) < 2^97 carries at most 1 into c, so
    // c <= e4 + 1 <= 2^32 - 2
    u32 e0 = (u32)a.e01, e1 = (u32)(a.e01 >> 32), e2 = (u32)a.e23, e3 = (u32)(a.e23 >> 32), c = a.e4;
    const u32 o0 = (u32)a.o01, o1 = (u32)(a.o01 >> 32);
    asm("add.cc.u32 %0, %0, %4; addc.cc.u32 %1, %1, %5; addc.cc.u32 %2, %2, %6; addc.u32 %3, %3, 0;"
        : "+r"(e1), "+r"(e2), "+r"(e3), "+r"(c) : "r"(o0), "r"(o1), "r"(a.o2));
    const u64 lo = e0 | ((u64)e1 << 32);
    const u64 s1 = e3 | ((u64)c << 32);  // hi_hi + c * 2^32 <= (2^32 - 2) 2^32 + 2^32 - 1 = p - 2: canonical, as gl_sub_cs needs
    u64 t0 = gl_sub_cs(lo, s1);
    const u64 t1 = ((u64)e2 << 32) - e2;  // hi_lo * (2^32 - 1) <= 2^64 - 2^33 + 1
    u64 r;
    u32 cy;
    asm("add.cc.u64 %0, %2, %3; addc.u32 %1, 0, 0;" : "=l"(r), "=r"(cy) : "l"(t0), "l"(t1));
    // on a carry r = t0 + t1 - 2^64 <= t1 - 1 <= 2^64 - 2^33, so r + EPS < 2^64 - 2^32 < p cannot wrap twice
    r += (u64)(0u - cy);
    return gl_canon(r);  // r < 2^64 < 2p: one conditional subtract makes it canonical
}
// extension-field accumulator: sum of products x*y kept as three unreduced base accumulators
struct xacc {
    acc192 a00, a11, ax;
};
__device__ __forceinline__ xacc xacc_zero() { xacc a; a.a00 = acc_zero(); a.a11 = acc_zero(); a.ax = acc_zero(); return a; }
__device__ __forceinline__ void xacc_mad(xacc& a, gl2 x, gl2 y) {
    acc_mad(a.a00, x.c0, y.c0);
    acc_mad(a.a11, x.c1, y.c1);
    acc_mad(a.ax, x.c0, y.c1);
    acc_mad(a.ax, x.c1, y.c0);
}
__device__ __forceinline__ void xacc_mad_base(xacc& a, gl2 x, u64 y) {
    acc_mad(a.a00, x.c0, y);
    acc_mad(a.ax, x.c1, y);
}
__device__ __forceinline__ gl2 xacc_reduce(const xacc& a) {
    acc192 t = a.a00;
    acc_mad(t, acc_reduce(a.a11), 7);  // X^2 = 7
    return gl2_make(acc_reduce(t), acc_reduce(a.ax));
}
// fold: a0 + r * (a1 - a0), canonical inputs, canonical output; r7 = 7 * r.c1 mod p
__device__ __forceinline__ gl2 gl2_fold(gl2 a0, gl2 a1, gl2 r, u64 r7) {
    const u64 d0 = gl_sub_cs(a1.c0, a0.c0), d1 = gl_sub_cs(a1.c1, a0.c1);
    acc192 c0 = acc_from(a0.c0), c1 = acc_from(a0.c1);
    acc_mad(c0, r.c0, d0);
    acc_mad(c0, r7, d1);
    acc_mad(c1, r.c0, d1);
    acc_mad(c1, r.c1, d0);
    return gl2_make(acc_reduce(c0), acc_reduce(c1));
}
__device__ __forceinline__ gl2 gl2_fold(u64 a0, u64 a1, gl2 r, u64) {
    const u64 d = gl_sub_cs(a1, a0);
    acc192 c0 = acc_from(a0), c1 = acc_zero();
    acc_mad(c0, r.c0, d);
    acc_mad(c1, r.c1, d);
    return gl2_make(acc_reduce(c0), acc_reduce(c1));
}
// canonical product of two canonical/lazy extension elements
__device__ __forceinline__ gl2 gl2_mul_fast(gl2 x, gl2 y) {
    xacc a = xacc_zero();
    xacc_mad(a, x, y);
    return xacc_reduce(a);
}
__device__ __forceinline__ u64 gl_mul_fast(u64 x, u64 y) {
    acc192 a = acc_zero();
    acc_mad(a, x, y);
    return acc_reduce(a);
}
#endif

}  // namespace hg
