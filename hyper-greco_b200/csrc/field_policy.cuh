// Field policies the kernels are templated on: base element B (tables as witnessed), extension element X
// (tables after the first fold, challenges, round messages).
//   GlField : B = Goldilocks u64, X = GoldilocksExt2 (16 B, one 128-bit load)
//   (BN254 Fr policy lives in bn254.cuh: B = X = 4x64 Montgomery)
#pragma once
#include <cstddef>

#include "gl.cuh"

namespace hg {

struct GlField {
    typedef u64 B;
    typedef gl2 X;
    static constexpr int FIELD_ID = 0;
    static constexpr int B_LIMBS = 1, X_LIMBS = 2;
    HG_HD static B b_zero() { return 0; }
    HG_HD static B b_one() { return 1; }
    HG_HD static B b_from_u64(u64 x) { return gl_from_u64(x); }
    HG_HD static B b_add(B a, B b) { return gl_add(a, b); }
    HG_HD static B b_sub(B a, B b) { return gl_sub(a, b); }
    HG_HD static B b_mul(B a, B b) { return gl_mul(a, b); }
    HG_HD static B b_inv(B a) { return gl_inv(a); }
    HG_HD static B root_of_unity() { return 0x185629dcda58878cULL; }  // 7^((p-1)/2^32), goldilocks ROOT_OF_UNITY (A9)
    static constexpr int TWO_ADICITY = 32;
    static constexpr int PLANES = 2;  // base planes per extension element
    static constexpr int GP_TAIL_LOG = 7, GP_MIN_BLOCKS = 2, GP_BLOCK = 128;
    static constexpr int GP_FOLD_CTAS = 4;      // CTAs of GP_BLOCK threads per SM the fold kernels are compiled for (5: 96 registers, 430-530 B of spills, GP class 1.97 instead of 1.66 ms)
    static constexpr int FUSED_MIN_BLOCKS = 4;  // CTAs of HG_FUSED_BLOCK threads per SM the fused tree builders are compiled for (gp_fused.cuh)
    static constexpr int GP_TAIL_GROUPS = 8;    // CTAs a layer is split over (by terms) in the tail kernel (profiles/r2_experiments.md)
    static constexpr int GP_BALANCE = 1;        // work-balanced term groups in the batched layer sumchecks (prover.cuh run_gp_batch)
    static constexpr double GP_TARGET = 0.25;  // CTAs per SM (of 256 threads) from which a layer runs with one term group (prover.cuh)
    HG_HD static bool b_eq(B a, B b) { return a == b; }
    HG_HD static B plane(X a, int p) { return p ? a.c1 : a.c0; }
    HG_HD static X from_planes(const B* p) { return gl2_make(p[0], p[1]); }
    HG_HD static X x_zero() { return gl2_zero(); }
    HG_HD static X x_one() { return gl2_one(); }
    HG_HD static X lift(B a) { return gl2_lift(a); }
    HG_HD static X x_add(X a, X b) { return gl2_add(a, b); }
    HG_HD static X x_sub(X a, X b) { return gl2_sub(a, b); }
    HG_HD static X x_mul(X a, X b) { return gl2_mul(a, b); }
    HG_HD static X x_mul_b(X a, B b) { return gl2_mul_base(a, b); }
    HG_HD static X x_add_b(X a, B b) { return gl2_make(gl_add(a.c0, b), a.c1); }
    HG_HD static bool x_eq(X a, X b) { return gl2_eq(a, b); }
    HG_HD static X x_inv(X a) { return gl2_inv(a); }
    HG_HD static B x_base0(X a) { return a.c0; }  // E::as_bases()[0], prover.rs:38-39
    // overloads so kernels can be written once for base or extension inputs
    HG_HD static X as_x(B a) { return gl2_lift(a); }
    HG_HD static X as_x(X a) { return a; }
    HG_HD static B sub(B a, B b) { return gl_sub(a, b); }
    HG_HD static X sub(X a, X b) { return gl2_sub(a, b); }
    HG_HD static B add(B a, B b) { return gl_add(a, b); }
    HG_HD static X add(X a, X b) { return gl2_add(a, b); }
    HG_HD static B mul(B a, B b) { return gl_mul(a, b); }
    HG_HD static X mul(X a, X b) { return gl2_mul(a, b); }
    HG_HD static X mul(X a, B b) { return gl2_mul_base(a, b); }
    HG_HD static X mul(B a, X b) { return gl2_mul_base(b, a); }
    HG_HD static u64 b_low_u64(B a) { return a; }  // low 64 bits of the canonical repr (fe_to_bits_le, lasso.rs:654-669)
    HG_HD static bool b_fits_u64(B) { return true; }
    // ---- host-side representation (transcript.rs:183-203; SURVEY Appendix B A1, A2, A11)
    typedef B Base;
    typedef X Ext;
    static constexpr int DEGREE = 2, REPR_BYTES = 8;
    static B base_from_le_bytes_mod(const unsigned char* h, size_t n) {  // fe_mod_from_le_bytes
        B acc = 0;
        for (size_t i = n; i-- > 0;) acc = gl_add(gl_mul(acc, 256), h[i]);
        return acc;
    }
    static void base_to_repr_le(B f, unsigned char* out) { for (int i = 0; i < 8; i++) out[i] = (unsigned char)(f >> (8 * i)); }
    static bool base_from_repr_le(const unsigned char* in, B* out) {
        u64 x = 0;
        for (int i = 0; i < 8; i++) x |= (u64)in[i] << (8 * i);
        if (x >= GL_P) return false;
        *out = x;
        return true;
    }
    static X ext_from_bases(const B* b) { return gl2_make(b[0], b[1]); }
    static void ext_as_bases(X e, B* b) { b[0] = e.c0; b[1] = e.c1; }
    // canonical u64 limbs at the C ABI
    static void b_to_limbs(B a, u64* out) { out[0] = a; }
    static B b_from_limbs(const u64* in) { return gl_from_u64(in[0]); }
    static void x_to_limbs(X a, u64* out) { out[0] = a.c0; out[1] = a.c1; }
    static X x_from_limbs(const u64* in) { return gl2_make(gl_from_u64(in[0]), gl_from_u64(in[1])); }
#if defined(__CUDACC__)
    __device__ __forceinline__ static X x_shfl_down(X v, int off) {
        return gl2_make(__shfl_down_sync(0xffffffffu, v.c0, off), __shfl_down_sync(0xffffffffu, v.c1, off));
    }
    // ---- fast device path (gl.cuh): lazy accumulators, canonical memory
    typedef acc192 BAcc;
    typedef xacc XAcc;
    struct FoldAux { u64 r7; };  // 7 * r.c1
    __device__ __forceinline__ static FoldAux fold_aux(X r) { FoldAux a; a.r7 = gl_mul7(r.c1); return a; }
    __device__ __forceinline__ static BAcc bacc_zero() { return acc_zero(); }
    __device__ __forceinline__ static void bacc_mad(BAcc& a, B x, B y) { acc_mad(a, x, y); }
    __device__ __forceinline__ static void bacc_add(BAcc& a, B x) { acc_add(a, x); }
    __device__ __forceinline__ static B b_shfl_down(B v, int off) { return __shfl_down_sync(0xffffffffu, v, off); }
    __device__ __forceinline__ static B bacc_reduce(const BAcc& a) { return acc_reduce(a); }
    __device__ __forceinline__ static XAcc xacc_zero_() { return xacc_zero(); }
    __device__ __forceinline__ static void xacc_mad_(XAcc& a, X x, X y) { xacc_mad(a, x, y); }
    __device__ __forceinline__ static void xacc_mad_b(XAcc& a, X x, B y) { xacc_mad_base(a, x, y); }
    __device__ __forceinline__ static X xacc_reduce_(const XAcc& a) { return xacc_reduce(a); }
    __device__ __forceinline__ static void xacc_mad_any(XAcc& a, X x, X y) { xacc_mad(a, x, y); }
    __device__ __forceinline__ static void xacc_mad_any(XAcc& a, X x, B y) { xacc_mad_base(a, x, y); }
    __device__ __forceinline__ static B fmul(B x, B y) { return gl_mul_fast(x, y); }
    __device__ __forceinline__ static X fmul(X x, X y) { return gl2_mul_fast(x, y); }
    __device__ __forceinline__ static X fmul_any(X x, X y) { return gl2_mul_fast(x, y); }
    __device__ __forceinline__ static X fmul_any(X x, B y) {  // extension * base: two products
        acc192 c0 = acc_zero(), c1 = acc_zero();
        acc_mad(c0, x.c0, y); acc_mad(c1, x.c1, y);
        return gl2_make(acc_reduce(c0), acc_reduce(c1));
    }
    // a0 + r (a1 - a0): canonical in, canonical out
    __device__ __forceinline__ static X fold(X a0, X a1, X r, FoldAux aux) { return gl2_fold(a0, a1, r, aux.r7); }
    __device__ __forceinline__ static X fold(B a0, B a1, X r, FoldAux aux) { return gl2_fold(a0, a1, r, aux.r7); }
    // c * (a0 + r (a1 - a0)) = c a0 + (c r)(a1 - a0) for base a0, a1 (round 1 of the grand product: fold + pre-scale)
    __device__ __forceinline__ static X fold_scaled(B a0, B a1, X c, X cr) {
        const u64 d = gl_sub_cs(a1, a0);
        acc192 c0 = acc_zero(), c1 = acc_zero();
        acc_mad(c0, c.c0, a0); acc_mad(c0, cr.c0, d);
        acc_mad(c1, c.c1, a0); acc_mad(c1, cr.c1, d);
        return gl2_make(acc_reduce(c0), acc_reduce(c1));
    }
    // line through (0, lo), (1, hi) at X = infinity (slope) and X = -1; canonical inputs, lazy outputs
    __device__ __forceinline__ static B slope(B lo, B hi) { return gl_sub_cs(hi, lo); }
    __device__ __forceinline__ static B at_m1(B lo, B hi) { return gl_add_cs(lo, gl_sub_cs(lo, hi)); }
    __device__ __forceinline__ static X slope(X lo, X hi) { return gl2_make(gl_sub_cs(hi.c0, lo.c0), gl_sub_cs(hi.c1, lo.c1)); }
    __device__ __forceinline__ static X at_m1(X lo, X hi) {
        return gl2_make(gl_add_cs(lo.c0, gl_sub_cs(lo.c0, hi.c0)), gl_add_cs(lo.c1, gl_sub_cs(lo.c1, hi.c1)));
    }
    // 2 q0 - q1 + 2 qinf for canonical inputs; some 64-bit representative (the result only feeds a multiplication)
    __device__ __forceinline__ static B q_at_m1(B q0, B q1, B qinf) {
        const u64 w = gl_add_cs(q0, gl_sub_cs(q0, q1));  // canonical + canonical-or-lazy
        return gl_add_cs(qinf, gl_add_cs(qinf, w));
    }
    __device__ __forceinline__ static B to_base(unsigned short v) { return (B)v; }
    __device__ __forceinline__ static B to_base(unsigned int v) { return (B)v; }
    __device__ __forceinline__ static B to_base(B v) { return v; }
    __device__ __forceinline__ static X x_ldcg(const X* p) {
        ulonglong2 t = __ldcg(reinterpret_cast<const ulonglong2*>(p));
        return gl2_make(t.x, t.y);
    }
#endif
};

}  // namespace hg
