// BN254 scalar field Fr in 4x64-bit Montgomery form, host + device, and its field policy (B = X = Fr: for BN254 the reference
// runs with E = F, /root/reference/bfv-gkr/src/sk_encryption_circuit.rs:616-626). Replaces halo2curves 0.7.0 bn256::Fr
// (/root/reference/Cargo.toml:29). r = 0x30644e72e131a029b85045b68181585d2833e84879b9709143e1f593f0000001
// (/root/reference/scripts/circuit_sk.py:50), R = 2^256, INV = -r^{-1} mod 2^64, two-adicity 28 with ROOT_OF_UNITY = 7^((r-1)/2^28).
// Every kernel on this field is bound by the integer pipes (16 64x64 multiplies per field multiplication), not by HBM.
#pragma once
#include <cstddef>

#include "gl.cuh"

namespace hg {

struct __align__(16) fr {
    u64 l[4];
};

constexpr u64 FR_MOD0 = 0x43e1f593f0000001ULL, FR_MOD1 = 0x2833e84879b97091ULL, FR_MOD2 = 0xb85045b68181585dULL, FR_MOD3 = 0x30644e72e131a029ULL;
constexpr u64 FR_INV = 0xc2e1f593efffffffULL;
// R^2 mod r (to Montgomery), R mod r (= one)
constexpr u64 FR_R2_0 = 0x1bb8e645ae216da7ULL, FR_R2_1 = 0x53fe3ab1e35c59e3ULL, FR_R2_2 = 0x8c49833d53bb8085ULL, FR_R2_3 = 0x0216d0b17f4e44a5ULL;
constexpr u64 FR_ONE0 = 0xac96341c4ffffffbULL, FR_ONE1 = 0x36fc76959f60cd29ULL, FR_ONE2 = 0x666ea36f7879462eULL, FR_ONE3 = 0x0e0a77c19a07df2fULL;

HG_HD fr fr_make(u64 a, u64 b, u64 c, u64 d) { fr r; r.l[0] = a; r.l[1] = b; r.l[2] = c; r.l[3] = d; return r; }
HG_HD fr fr_zero() { return fr_make(0, 0, 0, 0); }
HG_HD fr fr_one() { return fr_make(FR_ONE0, FR_ONE1, FR_ONE2, FR_ONE3); }
HG_HD bool fr_eq(const fr& a, const fr& b) { return a.l[0] == b.l[0] && a.l[1] == b.l[1] && a.l[2] == b.l[2] && a.l[3] == b.l[3]; }
HG_HD u64 fr_modl(int i) { return i == 0 ? FR_MOD0 : i == 1 ? FR_MOD1 : i == 2 ? FR_MOD2 : FR_MOD3; }
HG_HD bool fr_geq_mod(const u64* a) {
    if (a[3] != FR_MOD3) return a[3] > FR_MOD3;
    if (a[2] != FR_MOD2) return a[2] > FR_MOD2;
    if (a[1] != FR_MOD1) return a[1] > FR_MOD1;
    return a[0] >= FR_MOD0;
}
HG_HD u64 addc64(u64 a, u64 b, u64& carry) {  // a + b + carry
    u64 s = a + b;
    u64 c1 = s < a;
    u64 t = s + carry;
    carry = c1 | (u64)(t < s);
    return t;
}
HG_HD u64 subb64(u64 a, u64 b, u64& borrow) {  // a - b - borrow
    u64 d = a - b;
    u64 b1 = a < b;
    u64 t = d - borrow;
    borrow = b1 | (u64)(d < borrow);
    return t;
}
HG_HD void fr_sub_mod_inplace(u64* a) {
    u64 bw = 0;
    a[0] = subb64(a[0], FR_MOD0, bw); a[1] = subb64(a[1], FR_MOD1, bw); a[2] = subb64(a[2], FR_MOD2, bw); a[3] = subb64(a[3], FR_MOD3, bw);
}
#if defined(__CUDACC__)
// ---- device arithmetic with PTX carry chains (the portable C below compiles to compare/select sequences: 724 vs 481
// instructions per multiplication). Same results: Montgomery CIOS, fully reduced outputs.
// Contracts (raw Montgomery limbs; tests/test_field_probe.py checks each one at its boundaries):
//   fr_cond_sub_dev(t)           t < 2r as 5 limbs; output t mod r (t == r gives 0).
//   fr_add_dev, fr_sub_dev       a, b < r; output < r. No input may be lazy: a + b < 2r < 2^255 is what fr_cond_sub_dev takes.
//   fr_mul_dev, fr_mul_dev32     a, b < r; output a b R^-1 mod r, < r. In fr_mul_dev the running value stays below 2r, so
//                                t + a b_i + m r < 2^65 r < 2^320 never carries into t5 (r < 2^254): t5 and the t4 handed to
//                                fr_cond_sub_dev are 0 for inputs in contract.
__device__ __forceinline__ fr fr_cond_sub_dev(u64 t0, u64 t1, u64 t2, u64 t3, u64 t4) {  // (t4:t3:t2:t1:t0) < 2r  ->  mod r
    u64 s0, s1, s2, s3, bw;
    asm("sub.cc.u64 %0, %5, %9; subc.cc.u64 %1, %6, %10; subc.cc.u64 %2, %7, %11; subc.cc.u64 %3, %8, %12; subc.u64 %4, %13, 0;"
        : "=l"(s0), "=l"(s1), "=l"(s2), "=l"(s3), "=l"(bw)
        : "l"(t0), "l"(t1), "l"(t2), "l"(t3), "l"(FR_MOD0), "l"(FR_MOD1), "l"(FR_MOD2), "l"(FR_MOD3), "l"(t4));
    const bool keep = (bw >> 63) != 0;  // borrow out of the 5-limb subtraction: t < r
    fr r;
    r.l[0] = keep ? t0 : s0; r.l[1] = keep ? t1 : s1; r.l[2] = keep ? t2 : s2; r.l[3] = keep ? t3 : s3;
    return r;
}
__device__ __forceinline__ fr fr_add_dev(const fr& a, const fr& b) {
    u64 t0, t1, t2, t3;
    asm("add.cc.u64 %0, %4, %8; addc.cc.u64 %1, %5, %9; addc.cc.u64 %2, %6, %10; addc.u64 %3, %7, %11;"
        : "=l"(t0), "=l"(t1), "=l"(t2), "=l"(t3)
        : "l"(a.l[0]), "l"(a.l[1]), "l"(a.l[2]), "l"(a.l[3]), "l"(b.l[0]), "l"(b.l[1]), "l"(b.l[2]), "l"(b.l[3]));
    return fr_cond_sub_dev(t0, t1, t2, t3, 0);  // a + b < 2^255: no carry out of limb 3
}
__device__ __forceinline__ fr fr_sub_dev(const fr& a, const fr& b) {
    u64 t0, t1, t2, t3, bw;
    asm("sub.cc.u64 %0, %5, %9; subc.cc.u64 %1, %6, %10; subc.cc.u64 %2, %7, %11; subc.cc.u64 %3, %8, %12; subc.u64 %4, 0, 0;"
        : "=l"(t0), "=l"(t1), "=l"(t2), "=l"(t3), "=l"(bw)
        : "l"(a.l[0]), "l"(a.l[1]), "l"(a.l[2]), "l"(a.l[3]), "l"(b.l[0]), "l"(b.l[1]), "l"(b.l[2]), "l"(b.l[3]));
    // bw = 0 or all ones: add r masked
    asm("add.cc.u64 %0, %0, %4; addc.cc.u64 %1, %1, %5; addc.cc.u64 %2, %2, %6; addc.u64 %3, %3, %7;"
        : "+l"(t0), "+l"(t1), "+l"(t2), "+l"(t3) : "l"(FR_MOD0 & bw), "l"(FR_MOD1 & bw), "l"(FR_MOD2 & bw), "l"(FR_MOD3 & bw));
    fr r;
    r.l[0] = t0; r.l[1] = t1; r.l[2] = t2; r.l[3] = t3;
    return r;
}
__device__ __forceinline__ fr fr_mul_dev(const fr& a, const fr& b) {
    u64 t0 = 0, t1 = 0, t2 = 0, t3 = 0, t4 = 0, t5 = 0;
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const u64 bi = b.l[i];
        asm("{\n\t.reg .u64 m;\n\t"
            "mad.lo.cc.u64  %0, %6, %10, %0;\n\t"
            "madc.lo.cc.u64 %1, %7, %10, %1;\n\t"
            "madc.lo.cc.u64 %2, %8, %10, %2;\n\t"
            "madc.lo.cc.u64 %3, %9, %10, %3;\n\t"
            "addc.cc.u64    %4, %4, 0;\n\t"
            "addc.u64       %5, 0, 0;\n\t"
            "mad.hi.cc.u64  %1, %6, %10, %1;\n\t"
            "madc.hi.cc.u64 %2, %7, %10, %2;\n\t"
            "madc.hi.cc.u64 %3, %8, %10, %3;\n\t"
            "madc.hi.cc.u64 %4, %9, %10, %4;\n\t"
            "addc.u64       %5, %5, 0;\n\t"
            "mul.lo.u64     m, %0, %11;\n\t"
            "mad.lo.cc.u64  %0, m, %12, %0;\n\t"
            "madc.lo.cc.u64 %1, m, %13, %1;\n\t"
            "madc.lo.cc.u64 %2, m, %14, %2;\n\t"
            "madc.lo.cc.u64 %3, m, %15, %3;\n\t"
            "addc.cc.u64    %4, %4, 0;\n\t"
            "addc.u64       %5, %5, 0;\n\t"
            "mad.hi.cc.u64  %1, m, %12, %1;\n\t"
            "madc.hi.cc.u64 %2, m, %13, %2;\n\t"
            "madc.hi.cc.u64 %3, m, %14, %3;\n\t"
            "madc.hi.cc.u64 %4, m, %15, %4;\n\t"
            "addc.u64       %5, %5, 0;\n\t}"
            : "+l"(t0), "+l"(t1), "+l"(t2), "+l"(t3), "+l"(t4), "+l"(t5)
            : "l"(a.l[0]), "l"(a.l[1]), "l"(a.l[2]), "l"(a.l[3]), "l"(bi), "l"(FR_INV), "l"(FR_MOD0), "l"(FR_MOD1), "l"(FR_MOD2), "l"(FR_MOD3));
        t0 = t1; t1 = t2; t2 = t3; t3 = t4; t4 = t5; t5 = 0;  // the low limb is zero after the reduction step
    }
    return fr_cond_sub_dev(t0, t1, t2, t3, t4);
}
// 8 x 32-bit Montgomery multiplication with even / odd column accumulators (generated by scripts/gen_fr_mul.py, which also
// simulates the instruction list bit for bit against a * b * R^-1 mod r on random and extreme operands): the low and high half of
// every 32x32 product land on an ALIGNED register pair, so each mad.lo.cc / madc.hi.cc pair is one IMAD.WIDE.U32 with carry in
// SASS; the accumulator is divided by 2^32 per multiplier word by swapping the roles of the two column sets instead of moving
// registers. 294 PTX instructions (about 170 in SASS) against 481 for the 4 x 64-bit CIOS above. Result < 2r in e0..e7.
__device__ __forceinline__ fr fr_mul_dev32(const fr& a, const fr& b) {
    u64 r0, r1, r2, r3;
    asm("{\n\t"
        ".reg .u32 a0, a1, a2, a3, a4, a5, a6, a7, b0, b1, b2, b3, b4, b5, b6, b7;\n\t"
        ".reg .u32 e0, e1, e2, e3, e4, e5, e6, e7, o0, o1, o2, o3, o4, o5, o6, o7, mi;\n\t"
        "mov.b64 {a0, a1}, %4;\n\tmov.b64 {a2, a3}, %5;\n\tmov.b64 {a4, a5}, %6;\n\tmov.b64 {a6, a7}, %7;\n\t"
        "mov.b64 {b0, b1}, %8;\n\tmov.b64 {b2, b3}, %9;\n\tmov.b64 {b4, b5}, %10;\n\tmov.b64 {b6, b7}, %11;\n\t"
        "mul.lo.u32 o0, a1, b0;\n\t"
        "mul.hi.u32 o1, a1, b0;\n\t"
        "mul.lo.u32 o2, a3, b0;\n\t"
        "mul.hi.u32 o3, a3, b0;\n\t"
        "mul.lo.u32 o4, a5, b0;\n\t"
        "mul.hi.u32 o5, a5, b0;\n\t"
        "mul.lo.u32 o6, a7, b0;\n\t"
        "mul.hi.u32 o7, a7, b0;\n\t"
        "mul.lo.u32 e0, a0, b0;\n\t"
        "mul.hi.u32 e1, a0, b0;\n\t"
        "mul.lo.u32 e2, a2, b0;\n\t"
        "mul.hi.u32 e3, a2, b0;\n\t"
        "mul.lo.u32 e4, a4, b0;\n\t"
        "mul.hi.u32 e5, a4, b0;\n\t"
        "mul.lo.u32 e6, a6, b0;\n\t"
        "mul.hi.u32 e7, a6, b0;\n\t"
        "mul.lo.u32 mi, e0, 0xefffffff;\n\t"
        "mad.lo.cc.u32 o0, 0x43e1f593, mi, o0;\n\t"
        "madc.hi.cc.u32 o1, 0x43e1f593, mi, o1;\n\t"
        "madc.lo.cc.u32 o2, 0x2833e848, mi, o2;\n\t"
        "madc.hi.cc.u32 o3, 0x2833e848, mi, o3;\n\t"
        "madc.lo.cc.u32 o4, 0xb85045b6, mi, o4;\n\t"
        "madc.hi.cc.u32 o5, 0xb85045b6, mi, o5;\n\t"
        "madc.lo.cc.u32 o6, 0x30644e72, mi, o6;\n\t"
        "madc.hi.cc.u32 o7, 0x30644e72, mi, o7;\n\t"
        "mad.lo.cc.u32 e0, 0xf0000001, mi, e0;\n\t"
        "madc.hi.cc.u32 e1, 0xf0000001, mi, e1;\n\t"
        "madc.lo.cc.u32 e2, 0x79b97091, mi, e2;\n\t"
        "madc.hi.cc.u32 e3, 0x79b97091, mi, e3;\n\t"
        "madc.lo.cc.u32 e4, 0x8181585d, mi, e4;\n\t"
        "madc.hi.cc.u32 e5, 0x8181585d, mi, e5;\n\t"
        "madc.lo.cc.u32 e6, 0xe131a029, mi, e6;\n\t"
        "madc.hi.cc.u32 e7, 0xe131a029, mi, e7;\n\t"
        "addc.u32 o7, o7, 0;\n\t"
        "add.cc.u32 o0, o0, e1;\n\t"
        "madc.lo.cc.u32 e0, a1, b1, e2;\n\t"
        "madc.hi.cc.u32 e1, a1, b1, e3;\n\t"
        "madc.lo.cc.u32 e2, a3, b1, e4;\n\t"
        "madc.hi.cc.u32 e3, a3, b1, e5;\n\t"
        "madc.lo.cc.u32 e4, a5, b1, e6;\n\t"
        "madc.hi.cc.u32 e5, a5, b1, e7;\n\t"
        "madc.lo.cc.u32 e6, a7, b1, 0;\n\t"
        "madc.hi.u32 e7, a7, b1, 0;\n\t"
        "mad.lo.cc.u32 o0, a0, b1, o0;\n\t"
        "madc.hi.cc.u32 o1, a0, b1, o1;\n\t"
        "madc.lo.cc.u32 o2, a2, b1, o2;\n\t"
        "madc.hi.cc.u32 o3, a2, b1, o3;\n\t"
        "madc.lo.cc.u32 o4, a4, b1, o4;\n\t"
        "madc.hi.cc.u32 o5, a4, b1, o5;\n\t"
        "madc.lo.cc.u32 o6, a6, b1, o6;\n\t"
        "madc.hi.cc.u32 o7, a6, b1, o7;\n\t"
        "addc.u32 e7, e7, 0;\n\t"
        "mul.lo.u32 mi, o0, 0xefffffff;\n\t"
        "mad.lo.cc.u32 e0, 0x43e1f593, mi, e0;\n\t"
        "madc.hi.cc.u32 e1, 0x43e1f593, mi, e1;\n\t"
        "madc.lo.cc.u32 e2, 0x2833e848, mi, e2;\n\t"
        "madc.hi.cc.u32 e3, 0x2833e848, mi, e3;\n\t"
        "madc.lo.cc.u32 e4, 0xb85045b6, mi, e4;\n\t"
        "madc.hi.cc.u32 e5, 0xb85045b6, mi, e5;\n\t"
        "madc.lo.cc.u32 e6, 0x30644e72, mi, e6;\n\t"
        "madc.hi.cc.u32 e7, 0x30644e72, mi, e7;\n\t"
        "mad.lo.cc.u32 o0, 0xf0000001, mi, o0;\n\t"
        "madc.hi.cc.u32 o1, 0xf0000001, mi, o1;\n\t"
        "madc.lo.cc.u32 o2, 0x79b97091, mi, o2;\n\t"
        "madc.hi.cc.u32 o3, 0x79b97091, mi, o3;\n\t"
        "madc.lo.cc.u32 o4, 0x8181585d, mi, o4;\n\t"
        "madc.hi.cc.u32 o5, 0x8181585d, mi, o5;\n\t"
        "madc.lo.cc.u32 o6, 0xe131a029, mi, o6;\n\t"
        "madc.hi.cc.u32 o7, 0xe131a029, mi, o7;\n\t"
        "addc.u32 e7, e7, 0;\n\t"
        "add.cc.u32 e0, e0, o1;\n\t"
        "madc.lo.cc.u32 o0, a1, b2, o2;\n\t"
        "madc.hi.cc.u32 o1, a1, b2, o3;\n\t"
        "madc.lo.cc.u32 o2, a3, b2, o4;\n\t"
        "madc.hi.cc.u32 o3, a3, b2, o5;\n\t"
        "madc.lo.cc.u32 o4, a5, b2, o6;\n\t"
        "madc.hi.cc.u32 o5, a5, b2, o7;\n\t"
        "madc.lo.cc.u32 o6, a7, b2, 0;\n\t"
        "madc.hi.u32 o7, a7, b2, 0;\n\t"
        "mad.lo.cc.u32 e0, a0, b2, e0;\n\t"
        "madc.hi.cc.u32 e1, a0, b2, e1;\n\t"
        "madc.lo.cc.u32 e2, a2, b2, e2;\n\t"
        "madc.hi.cc.u32 e3, a2, b2, e3;\n\t"
        "madc.lo.cc.u32 e4, a4, b2, e4;\n\t"
        "madc.hi.cc.u32 e5, a4, b2, e5;\n\t"
        "madc.lo.cc.u32 e6, a6, b2, e6;\n\t"
        "madc.hi.cc.u32 e7, a6, b2, e7;\n\t"
        "addc.u32 o7, o7, 0;\n\t"
        "mul.lo.u32 mi, e0, 0xefffffff;\n\t"
        "mad.lo.cc.u32 o0, 0x43e1f593, mi, o0;\n\t"
        "madc.hi.cc.u32 o1, 0x43e1f593, mi, o1;\n\t"
        "madc.lo.cc.u32 o2, 0x2833e848, mi, o2;\n\t"
        "madc.hi.cc.u32 o3, 0x2833e848, mi, o3;\n\t"
        "madc.lo.cc.u32 o4, 0xb85045b6, mi, o4;\n\t"
        "madc.hi.cc.u32 o5, 0xb85045b6, mi, o5;\n\t"
        "madc.lo.cc.u32 o6, 0x30644e72, mi, o6;\n\t"
        "madc.hi.cc.u32 o7, 0x30644e72, mi, o7;\n\t"
        "mad.lo.cc.u32 e0, 0xf0000001, mi, e0;\n\t"
        "madc.hi.cc.u32 e1, 0xf0000001, mi, e1;\n\t"
        "madc.lo.cc.u32 e2, 0x79b97091, mi, e2;\n\t"
        "madc.hi.cc.u32 e3, 0x79b97091, mi, e3;\n\t"
        "madc.lo.cc.u32 e4, 0x8181585d, mi, e4;\n\t"
        "madc.hi.cc.u32 e5, 0x8181585d, mi, e5;\n\t"
        "madc.lo.cc.u32 e6, 0xe131a029, mi, e6;\n\t"
        "madc.hi.cc.u32 e7, 0xe131a029, mi, e7;\n\t"
        "addc.u32 o7, o7, 0;\n\t"
        "add.cc.u32 o0, o0, e1;\n\t"
        "madc.lo.cc.u32 e0, a1, b3, e2;\n\t"
        "madc.hi.cc.u32 e1, a1, b3, e3;\n\t"
        "madc.lo.cc.u32 e2, a3, b3, e4;\n\t"
        "madc.hi.cc.u32 e3, a3, b3, e5;\n\t"
        "madc.lo.cc.u32 e4, a5, b3, e6;\n\t"
        "madc.hi.cc.u32 e5, a5, b3, e7;\n\t"
        "madc.lo.cc.u32 e6, a7, b3, 0;\n\t"
        "madc.hi.u32 e7, a7, b3, 0;\n\t"
        "mad.lo.cc.u32 o0, a0, b3, o0;\n\t"
        "madc.hi.cc.u32 o1, a0, b3, o1;\n\t"
        "madc.lo.cc.u32 o2, a2, b3, o2;\n\t"
        "madc.hi.cc.u32 o3, a2, b3, o3;\n\t"
        "madc.lo.cc.u32 o4, a4, b3, o4;\n\t"
        "madc.hi.cc.u32 o5, a4, b3, o5;\n\t"
        "madc.lo.cc.u32 o6, a6, b3, o6;\n\t"
        "madc.hi.cc.u32 o7, a6, b3, o7;\n\t"
        "addc.u32 e7, e7, 0;\n\t"
        "mul.lo.u32 mi, o0, 0xefffffff;\n\t"
        "mad.lo.cc.u32 e0, 0x43e1f593, mi, e0;\n\t"
        "madc.hi.cc.u32 e1, 0x43e1f593, mi, e1;\n\t"
        "madc.lo.cc.u32 e2, 0x2833e848, mi, e2;\n\t"
        "madc.hi.cc.u32 e3, 0x2833e848, mi, e3;\n\t"
        "madc.lo.cc.u32 e4, 0xb85045b6, mi, e4;\n\t"
        "madc.hi.cc.u32 e5, 0xb85045b6, mi, e5;\n\t"
        "madc.lo.cc.u32 e6, 0x30644e72, mi, e6;\n\t"
        "madc.hi.cc.u32 e7, 0x30644e72, mi, e7;\n\t"
        "mad.lo.cc.u32 o0, 0xf0000001, mi, o0;\n\t"
        "madc.hi.cc.u32 o1, 0xf0000001, mi, o1;\n\t"
        "madc.lo.cc.u32 o2, 0x79b97091, mi, o2;\n\t"
        "madc.hi.cc.u32 o3, 0x79b97091, mi, o3;\n\t"
        "madc.lo.cc.u32 o4, 0x8181585d, mi, o4;\n\t"
        "madc.hi.cc.u32 o5, 0x8181585d, mi, o5;\n\t"
        "madc.lo.cc.u32 o6, 0xe131a029, mi, o6;\n\t"
        "madc.hi.cc.u32 o7, 0xe131a029, mi, o7;\n\t"
        "addc.u32 e7, e7, 0;\n\t"
        "add.cc.u32 e0, e0, o1;\n\t"
        "madc.lo.cc.u32 o0, a1, b4, o2;\n\t"
        "madc.hi.cc.u32 o1, a1, b4, o3;\n\t"
        "madc.lo.cc.u32 o2, a3, b4, o4;\n\t"
        "madc.hi.cc.u32 o3, a3, b4, o5;\n\t"
        "madc.lo.cc.u32 o4, a5, b4, o6;\n\t"
        "madc.hi.cc.u32 o5, a5, b4, o7;\n\t"
        "madc.lo.cc.u32 o6, a7, b4, 0;\n\t"
        "madc.hi.u32 o7, a7, b4, 0;\n\t"
        "mad.lo.cc.u32 e0, a0, b4, e0;\n\t"
        "madc.hi.cc.u32 e1, a0, b4, e1;\n\t"
        "madc.lo.cc.u32 e2, a2, b4, e2;\n\t"
        "madc.hi.cc.u32 e3, a2, b4, e3;\n\t"
        "madc.lo.cc.u32 e4, a4, b4, e4;\n\t"
        "madc.hi.cc.u32 e5, a4, b4, e5;\n\t"
        "madc.lo.cc.u32 e6, a6, b4, e6;\n\t"
        "madc.hi.cc.u32 e7, a6, b4, e7;\n\t"
        "addc.u32 o7, o7, 0;\n\t"
        "mul.lo.u32 mi, e0, 0xefffffff;\n\t"
        "mad.lo.cc.u32 o0, 0x43e1f593, mi, o0;\n\t"
        "madc.hi.cc.u32 o1, 0x43e1f593, mi, o1;\n\t"
        "madc.lo.cc.u32 o2, 0x2833e848, mi, o2;\n\t"
        "madc.hi.cc.u32 o3, 0x2833e848, mi, o3;\n\t"
        "madc.lo.cc.u32 o4, 0xb85045b6, mi, o4;\n\t"
        "madc.hi.cc.u32 o5, 0xb85045b6, mi, o5;\n\t"
        "madc.lo.cc.u32 o6, 0x30644e72, mi, o6;\n\t"
        "madc.hi.cc.u32 o7, 0x30644e72, mi, o7;\n\t"
        "mad.lo.cc.u32 e0, 0xf0000001, mi, e0;\n\t"
        "madc.hi.cc.u32 e1, 0xf0000001, mi, e1;\n\t"
        "madc.lo.cc.u32 e2, 0x79b97091, mi, e2;\n\t"
        "madc.hi.cc.u32 e3, 0x79b97091, mi, e3;\n\t"
        "madc.lo.cc.u32 e4, 0x8181585d, mi, e4;\n\t"
        "madc.hi.cc.u32 e5, 0x8181585d, mi, e5;\n\t"
        "madc.lo.cc.u32 e6, 0xe131a029, mi, e6;\n\t"
        "madc.hi.cc.u32 e7, 0xe131a029, mi, e7;\n\t"
        "addc.u32 o7, o7, 0;\n\t"
        "add.cc.u32 o0, o0, e1;\n\t"
        "madc.lo.cc.u32 e0, a1, b5, e2;\n\t"
        "madc.hi.cc.u32 e1, a1, b5, e3;\n\t"
        "madc.lo.cc.u32 e2, a3, b5, e4;\n\t"
        "madc.hi.cc.u32 e3, a3, b5, e5;\n\t"
        "madc.lo.cc.u32 e4, a5, b5, e6;\n\t"
        "madc.hi.cc.u32 e5, a5, b5, e7;\n\t"
        "madc.lo.cc.u32 e6, a7, b5, 0;\n\t"
        "madc.hi.u32 e7, a7, b5, 0;\n\t"
        "mad.lo.cc.u32 o0, a0, b5, o0;\n\t"
        "madc.hi.cc.u32 o1, a0, b5, o1;\n\t"
        "madc.lo.cc.u32 o2, a2, b5, o2;\n\t"
        "madc.hi.cc.u32 o3, a2, b5, o3;\n\t"
        "madc.lo.cc.u32 o4, a4, b5, o4;\n\t"
        "madc.hi.cc.u32 o5, a4, b5, o5;\n\t"
        "madc.lo.cc.u32 o6, a6, b5, o6;\n\t"
        "madc.hi.cc.u32 o7, a6, b5, o7;\n\t"
        "addc.u32 e7, e7, 0;\n\t"
        "mul.lo.u32 mi, o0, 0xefffffff;\n\t"
        "mad.lo.cc.u32 e0, 0x43e1f593, mi, e0;\n\t"
        "madc.hi.cc.u32 e1, 0x43e1f593, mi, e1;\n\t"
        "madc.lo.cc.u32 e2, 0x2833e848, mi, e2;\n\t"
        "madc.hi.cc.u32 e3, 0x2833e848, mi, e3;\n\t"
        "madc.lo.cc.u32 e4, 0xb85045b6, mi, e4;\n\t"
        "madc.hi.cc.u32 e5, 0xb85045b6, mi, e5;\n\t"
        "madc.lo.cc.u32 e6, 0x30644e72, mi, e6;\n\t"
        "madc.hi.cc.u32 e7, 0x30644e72, mi, e7;\n\t"
        "mad.lo.cc.u32 o0, 0xf0000001, mi, o0;\n\t"
        "madc.hi.cc.u32 o1, 0xf0000001, mi, o1;\n\t"
        "madc.lo.cc.u32 o2, 0x79b97091, mi, o2;\n\t"
        "madc.hi.cc.u32 o3, 0x79b97091, mi, o3;\n\t"
        "madc.lo.cc.u32 o4, 0x8181585d, mi, o4;\n\t"
        "madc.hi.cc.u32 o5, 0x8181585d, mi, o5;\n\t"
        "madc.lo.cc.u32 o6, 0xe131a029, mi, o6;\n\t"
        "madc.hi.cc.u32 o7, 0xe131a029, mi, o7;\n\t"
        "addc.u32 e7, e7, 0;\n\t"
        "add.cc.u32 e0, e0, o1;\n\t"
        "madc.lo.cc.u32 o0, a1, b6, o2;\n\t"
        "madc.hi.cc.u32 o1, a1, b6, o3;\n\t"
        "madc.lo.cc.u32 o2, a3, b6, o4;\n\t"
        "madc.hi.cc.u32 o3, a3, b6, o5;\n\t"
        "madc.lo.cc.u32 o4, a5, b6, o6;\n\t"
        "madc.hi.cc.u32 o5, a5, b6, o7;\n\t"
        "madc.lo.cc.u32 o6, a7, b6, 0;\n\t"
        "madc.hi.u32 o7, a7, b6, 0;\n\t"
        "mad.lo.cc.u32 e0, a0, b6, e0;\n\t"
        "madc.hi.cc.u32 e1, a0, b6, e1;\n\t"
        "madc.lo.cc.u32 e2, a2, b6, e2;\n\t"
        "madc.hi.cc.u32 e3, a2, b6, e3;\n\t"
        "madc.lo.cc.u32 e4, a4, b6, e4;\n\t"
        "madc.hi.cc.u32 e5, a4, b6, e5;\n\t"
        "madc.lo.cc.u32 e6, a6, b6, e6;\n\t"
        "madc.hi.cc.u32 e7, a6, b6, e7;\n\t"
        "addc.u32 o7, o7, 0;\n\t"
        "mul.lo.u32 mi, e0, 0xefffffff;\n\t"
        "mad.lo.cc.u32 o0, 0x43e1f593, mi, o0;\n\t"
        "madc.hi.cc.u32 o1, 0x43e1f593, mi, o1;\n\t"
        "madc.lo.cc.u32 o2, 0x2833e848, mi, o2;\n\t"
        "madc.hi.cc.u32 o3, 0x2833e848, mi, o3;\n\t"
        "madc.lo.cc.u32 o4, 0xb85045b6, mi, o4;\n\t"
        "madc.hi.cc.u32 o5, 0xb85045b6, mi, o5;\n\t"
        "madc.lo.cc.u32 o6, 0x30644e72, mi, o6;\n\t"
        "madc.hi.cc.u32 o7, 0x30644e72, mi, o7;\n\t"
        "mad.lo.cc.u32 e0, 0xf0000001, mi, e0;\n\t"
        "madc.hi.cc.u32 e1, 0xf0000001, mi, e1;\n\t"
        "madc.lo.cc.u32 e2, 0x79b97091, mi, e2;\n\t"
        "madc.hi.cc.u32 e3, 0x79b97091, mi, e3;\n\t"
        "madc.lo.cc.u32 e4, 0x8181585d, mi, e4;\n\t"
        "madc.hi.cc.u32 e5, 0x8181585d, mi, e5;\n\t"
        "madc.lo.cc.u32 e6, 0xe131a029, mi, e6;\n\t"
        "madc.hi.cc.u32 e7, 0xe131a029, mi, e7;\n\t"
        "addc.u32 o7, o7, 0;\n\t"
        "add.cc.u32 o0, o0, e1;\n\t"
        "madc.lo.cc.u32 e0, a1, b7, e2;\n\t"
        "madc.hi.cc.u32 e1, a1, b7, e3;\n\t"
        "madc.lo.cc.u32 e2, a3, b7, e4;\n\t"
        "madc.hi.cc.u32 e3, a3, b7, e5;\n\t"
        "madc.lo.cc.u32 e4, a5, b7, e6;\n\t"
        "madc.hi.cc.u32 e5, a5, b7, e7;\n\t"
        "madc.lo.cc.u32 e6, a7, b7, 0;\n\t"
        "madc.hi.u32 e7, a7, b7, 0;\n\t"
        "mad.lo.cc.u32 o0, a0, b7, o0;\n\t"
        "madc.hi.cc.u32 o1, a0, b7, o1;\n\t"
        "madc.lo.cc.u32 o2, a2, b7, o2;\n\t"
        "madc.hi.cc.u32 o3, a2, b7, o3;\n\t"
        "madc.lo.cc.u32 o4, a4, b7, o4;\n\t"
        "madc.hi.cc.u32 o5, a4, b7, o5;\n\t"
        "madc.lo.cc.u32 o6, a6, b7, o6;\n\t"
        "madc.hi.cc.u32 o7, a6, b7, o7;\n\t"
        "addc.u32 e7, e7, 0;\n\t"
        "mul.lo.u32 mi, o0, 0xefffffff;\n\t"
        "mad.lo.cc.u32 e0, 0x43e1f593, mi, e0;\n\t"
        "madc.hi.cc.u32 e1, 0x43e1f593, mi, e1;\n\t"
        "madc.lo.cc.u32 e2, 0x2833e848, mi, e2;\n\t"
        "madc.hi.cc.u32 e3, 0x2833e848, mi, e3;\n\t"
        "madc.lo.cc.u32 e4, 0xb85045b6, mi, e4;\n\t"
        "madc.hi.cc.u32 e5, 0xb85045b6, mi, e5;\n\t"
        "madc.lo.cc.u32 e6, 0x30644e72, mi, e6;\n\t"
        "madc.hi.cc.u32 e7, 0x30644e72, mi, e7;\n\t"
        "mad.lo.cc.u32 o0, 0xf0000001, mi, o0;\n\t"
        "madc.hi.cc.u32 o1, 0xf0000001, mi, o1;\n\t"
        "madc.lo.cc.u32 o2, 0x79b97091, mi, o2;\n\t"
        "madc.hi.cc.u32 o3, 0x79b97091, mi, o3;\n\t"
        "madc.lo.cc.u32 o4, 0x8181585d, mi, o4;\n\t"
        "madc.hi.cc.u32 o5, 0x8181585d, mi, o5;\n\t"
        "madc.lo.cc.u32 o6, 0xe131a029, mi, o6;\n\t"
        "madc.hi.cc.u32 o7, 0xe131a029, mi, o7;\n\t"
        "addc.u32 e7, e7, 0;\n\t"
        "add.cc.u32 e0, e0, o1;\n\t"
        "addc.cc.u32 e1, e1, o2;\n\t"
        "addc.cc.u32 e2, e2, o3;\n\t"
        "addc.cc.u32 e3, e3, o4;\n\t"
        "addc.cc.u32 e4, e4, o5;\n\t"
        "addc.cc.u32 e5, e5, o6;\n\t"
        "addc.cc.u32 e6, e6, o7;\n\t"
        "addc.u32 e7, e7, 0;\n\t"
        "mov.b64 %0, {e0, e1};\n\tmov.b64 %1, {e2, e3};\n\tmov.b64 %2, {e4, e5};\n\tmov.b64 %3, {e6, e7};\n\t}"
        : "=l"(r0), "=l"(r1), "=l"(r2), "=l"(r3)
        : "l"(a.l[0]), "l"(a.l[1]), "l"(a.l[2]), "l"(a.l[3]), "l"(b.l[0]), "l"(b.l[1]), "l"(b.l[2]), "l"(b.l[3]));
    return fr_cond_sub_dev(r0, r1, r2, r3, 0);
}
#endif
HG_HD fr fr_add(const fr& a, const fr& b) {
#if defined(__CUDA_ARCH__)
    return fr_add_dev(a, b);
#else
    fr r;
    u64 c = 0;
    for (int i = 0; i < 4; i++) r.l[i] = addc64(a.l[i], b.l[i], c);
    if (c || fr_geq_mod(r.l)) fr_sub_mod_inplace(r.l);  // r < 2^254 so c is always 0; kept for clarity
    return r;
#endif
}
HG_HD fr fr_sub(const fr& a, const fr& b) {
#if defined(__CUDA_ARCH__)
    return fr_sub_dev(a, b);
#else
    fr r;
    u64 bw = 0;
    for (int i = 0; i < 4; i++) r.l[i] = subb64(a.l[i], b.l[i], bw);
    if (bw) { u64 c = 0; r.l[0] = addc64(r.l[0], FR_MOD0, c); r.l[1] = addc64(r.l[1], FR_MOD1, c); r.l[2] = addc64(r.l[2], FR_MOD2, c); r.l[3] = addc64(r.l[3], FR_MOD3, c); }
    return r;
#endif
}
// Montgomery product a * b * R^{-1} mod r (CIOS, 4 limbs)
HG_HD fr fr_mul(const fr& a, const fr& b) {
#if defined(__CUDA_ARCH__)
#if defined(HG_FR_MUL64)
    return fr_mul_dev(a, b);
#else
    return fr_mul_dev32(a, b);
#endif
#else
    u64 t[6] = {0, 0, 0, 0, 0, 0};
#pragma unroll
    for (int i = 0; i < 4; i++) {
        u64 carry = 0;
#pragma unroll
        for (int j = 0; j < 4; j++) {
            u64 lo, hi;
            mul_wide(a.l[j], b.l[i], lo, hi);
            u64 c = 0;
            u64 s = addc64(t[j], lo, c);
            hi += c;
            c = 0;
            s = addc64(s, carry, c);
            hi += c;
            t[j] = s;
            carry = hi;
        }
        u64 c = 0;
        t[4] = addc64(t[4], carry, c);
        t[5] = c;
        const u64 m = t[0] * FR_INV;
        u64 lo, hi;
        mul_wide(m, FR_MOD0, lo, hi);
        c = 0;
        (void)addc64(t[0], lo, c);
        carry = hi + c;
#pragma unroll
        for (int j = 1; j < 4; j++) {
            mul_wide(m, fr_modl(j), lo, hi);
            u64 c2 = 0;
            u64 s = addc64(t[j], lo, c2);
            hi += c2;
            c2 = 0;
            s = addc64(s, carry, c2);
            hi += c2;
            t[j - 1] = s;
            carry = hi;
        }
        c = 0;
        t[3] = addc64(t[4], carry, c);
        t[4] = t[5] + c;
    }
    fr r = fr_make(t[0], t[1], t[2], t[3]);
    if (t[4] || fr_geq_mod(r.l)) fr_sub_mod_inplace(r.l);
    return r;
#endif
}
HG_HD fr fr_from_canonical(const u64* x) { return fr_mul(fr_make(x[0], x[1], x[2], x[3]), fr_make(FR_R2_0, FR_R2_1, FR_R2_2, FR_R2_3)); }
HG_HD void fr_to_canonical(const fr& a, u64* out) {
    fr r = fr_mul(a, fr_make(1, 0, 0, 0));
    out[0] = r.l[0]; out[1] = r.l[1]; out[2] = r.l[2]; out[3] = r.l[3];
}
HG_HD fr fr_from_u64(u64 x) { u64 t[4] = {x, 0, 0, 0}; return fr_from_canonical(t); }
HG_HD fr fr_pow(fr b, const u64* e, int n) {
    fr r = fr_one();
    for (int i = 0; i < n; i++) for (int k = 0; k < 64; k++) { if ((e[i] >> k) & 1) r = fr_mul(r, b); b = fr_mul(b, b); }
    return r;
}
HG_HD fr fr_inv(const fr& a) {
    u64 e[4] = {FR_MOD0 - 2, FR_MOD1, FR_MOD2, FR_MOD3};
    return fr_pow(a, e, 4);
}

struct FrField {
    typedef fr B;
    typedef fr X;
    static constexpr int FIELD_ID = 1;
    static constexpr int B_LIMBS = 4, X_LIMBS = 4;
    static constexpr int PLANES = 1;  // base planes per extension element
    static constexpr int GP_TAIL_LOG = 5, GP_MIN_BLOCKS = 1, GP_BLOCK = 128;
    static constexpr int GP_FOLD_CTAS = 3;      // CTAs of GP_BLOCK threads per SM the fold kernels are compiled for
    static constexpr int FUSED_MIN_BLOCKS = 2;
    static constexpr int GP_TAIL_GROUPS = 4;
    static constexpr int GP_BALANCE = 0;
    static constexpr double GP_TARGET = 2.0;
    HG_HD static B b_zero() { return fr_zero(); }
    HG_HD static B b_one() { return fr_one(); }
    HG_HD static B b_from_u64(u64 x) { return fr_from_u64(x); }
    HG_HD static B b_add(B a, B b) { return fr_add(a, b); }
    HG_HD static B b_sub(B a, B b) { return fr_sub(a, b); }
    HG_HD static B b_mul(B a, B b) { return fr_mul(a, b); }
    HG_HD static B b_inv(B a) { return fr_inv(a); }
    HG_HD static bool b_eq(B a, B b) { return fr_eq(a, b); }
    static constexpr int TWO_ADICITY = 28;
    HG_HD static B root_of_unity() {  // 7^((r-1)/2^28) = halo2curves bn256::Fr::ROOT_OF_UNITY (A9)
        const u64 raw[4] = {0xd34f1ed960c37c9cULL, 0x3215cf6dd39329c8ULL, 0x98865ea93dd31f74ULL, 0x03ddb9f5166d18b7ULL};
        return fr_from_canonical(raw);
    }
    HG_HD static X x_zero() { return fr_zero(); }
    HG_HD static X x_one() { return fr_one(); }
    HG_HD static X lift(B a) { return a; }
    HG_HD static X x_add(X a, X b) { return fr_add(a, b); }
    HG_HD static X x_sub(X a, X b) { return fr_sub(a, b); }
    HG_HD static X x_mul(X a, X b) { return fr_mul(a, b); }
    HG_HD static X x_mul_b(X a, B b) { return fr_mul(a, b); }
    HG_HD static bool x_eq(X a, X b) { return fr_eq(a, b); }
    HG_HD static X x_inv(X a) { return fr_inv(a); }
    HG_HD static B x_base0(X a) { return a; }
    HG_HD static X as_x(B a) { return a; }
    HG_HD static B sub(B a, B b) { return fr_sub(a, b); }
    HG_HD static B add(B a, B b) { return fr_add(a, b); }
    HG_HD static B mul(B a, B b) { return fr_mul(a, b); }
    HG_HD static u64 b_low_u64(B a) { u64 t[4]; fr_to_canonical(a, t); return t[0]; }  // low 64 bits of the LE repr; higher bits are truncated by lasso.rs:389 (Q8)
    HG_HD static B plane(X a, int) { return a; }
    HG_HD static X from_planes(const B* p) { return p[0]; }
    // ---- host representation (transcript.rs:183-203; A1: canonical little-endian 32 bytes, A11: 256-bit LE integer mod r)
    typedef B Base;
    typedef X Ext;
    static constexpr int DEGREE = 1, REPR_BYTES = 32;
    static B base_from_le_bytes_mod(const unsigned char* h, size_t n) {
        B acc = fr_zero(), b256 = fr_from_u64(256);
        for (size_t i = n; i-- > 0;) acc = fr_add(fr_mul(acc, b256), fr_from_u64(h[i]));
        return acc;
    }
    static void base_to_repr_le(B f, unsigned char* out) {
        u64 t[4];
        fr_to_canonical(f, t);
        for (int i = 0; i < 32; i++) out[i] = (unsigned char)(t[i / 8] >> (8 * (i % 8)));
    }
    static bool base_from_repr_le(const unsigned char* in, B* out) {
        u64 t[4] = {0, 0, 0, 0};
        for (int i = 0; i < 32; i++) t[i / 8] |= (u64)in[i] << (8 * (i % 8));
        if (fr_geq_mod(t)) return false;
        *out = fr_from_canonical(t);
        return true;
    }
    static X ext_from_bases(const B* b) { return b[0]; }
    static void ext_as_bases(X e, B* b) { b[0] = e; }
    static void b_to_limbs(B a, u64* out) { fr_to_canonical(a, out); }
    static B b_from_limbs(const u64* in) { u64 t[4] = {in[0], in[1], in[2], in[3]}; while (fr_geq_mod(t)) fr_sub_mod_inplace(t); return fr_from_canonical(t); }
    static void x_to_limbs(X a, u64* out) { fr_to_canonical(a, out); }
    static X x_from_limbs(const u64* in) { return b_from_limbs(in); }
#if defined(__CUDACC__)
    __device__ __forceinline__ static X x_shfl_down(X v, int off) {
        X r;
#pragma unroll
        for (int i = 0; i < 4; i++) r.l[i] = __shfl_down_sync(0xffffffffu, v.l[i], off);
        return r;
    }
    __device__ __forceinline__ static X x_ldcg(const X* p) {
        const ulonglong2* q = reinterpret_cast<const ulonglong2*>(p);
        ulonglong2 a = __ldcg(q), b = __ldcg(q + 1);
        return fr_make(a.x, a.y, b.x, b.y);
    }
    // "accumulators" are plain field elements here: Fr has no cheap lazy reduction in 4x64 form
    typedef fr BAcc;
    typedef fr XAcc;
    struct FoldAux { int unused; };
    __device__ __forceinline__ static FoldAux fold_aux(X) { FoldAux a; a.unused = 0; return a; }
    __device__ __forceinline__ static BAcc bacc_zero() { return fr_zero(); }
    __device__ __forceinline__ static void bacc_mad(BAcc& a, B x, B y) { a = fr_add(a, fr_mul(x, y)); }
    __device__ __forceinline__ static void bacc_add(BAcc& a, B x) { a = fr_add(a, x); }
    __device__ __forceinline__ static B b_shfl_down(B v, int off) { return x_shfl_down(v, off); }
    __device__ __forceinline__ static B bacc_reduce(const BAcc& a) { return a; }
    __device__ __forceinline__ static XAcc xacc_zero_() { return fr_zero(); }
    __device__ __forceinline__ static void xacc_mad_(XAcc& a, X x, X y) { a = fr_add(a, fr_mul(x, y)); }
    __device__ __forceinline__ static void xacc_mad_b(XAcc& a, X x, B y) { a = fr_add(a, fr_mul(x, y)); }
    __device__ __forceinline__ static X xacc_reduce_(const XAcc& a) { return a; }
    __device__ __forceinline__ static void xacc_mad_any(XAcc& a, X x, X y) { a = fr_add(a, fr_mul(x, y)); }
    __device__ __forceinline__ static X fmul(X x, X y) { return fr_mul(x, y); }
    __device__ __forceinline__ static X fmul_any(X x, X y) { return fr_mul(x, y); }
    __device__ __forceinline__ static X fold(X a0, X a1, X r, FoldAux) { return fr_add(a0, fr_mul(r, fr_sub(a1, a0))); }
    __device__ __forceinline__ static X fold_scaled(B a0, B a1, X c, X cr) { return fr_add(fr_mul(c, a0), fr_mul(cr, fr_sub(a1, a0))); }
    __device__ __forceinline__ static X slope(X lo, X hi) { return fr_sub(hi, lo); }
    __device__ __forceinline__ static X at_m1(X lo, X hi) { return fr_sub(fr_add(lo, lo), hi); }
    __device__ __forceinline__ static B q_at_m1(B q0, B q1, B qinf) { const B s = fr_add(q0, qinf); return fr_sub(fr_add(s, s), q1); }
    __device__ __forceinline__ static B to_base(unsigned short v) { return fr_from_u64(v); }
    __device__ __forceinline__ static B to_base(unsigned int v) { return fr_from_u64(v); }
    __device__ __forceinline__ static B to_base(B v) { return v; }
#endif
};

}  // namespace hg
