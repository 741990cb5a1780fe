// Test-only device probe of the field primitives the hot kernels are built on (gl.cuh fast path, GlField in field_policy.cuh,
// the PTX carry chains of bn254.cuh). Not part of libhg_b200.so: tests/test_field_probe.py compiles it into a temporary
// directory and calls probe_run through ctypes. One case per thread; every case reads in_words and writes out_words u64.
#include <cuda_runtime.h>

#include "field_policy.cuh"
#include "bn254.cuh"

using namespace hg;

enum {
    OP_ACC_REDUCE = 0,  // in: e01 e23 o01 e4 o2                          out: acc_reduce
    OP_ACC_RUN = 1,     // in: e01 e23 o01 e4 o2 x y z reps                out: acc_reduce after reps x (acc_mad(x, y); acc_add(z))
    OP_XACC = 2,        // in: 3 x (e01 e23 o01 e4 o2) for a00 a11 ax, x(2) y(2) yb
                        // out: xacc_reduce after xacc_mad(x, y), xacc_mad_base(x, yb)   (2)
    OP_SUB_ADD = 3,     // in: a b    out: gl_sub_cs(a, b), gl_add_cs(b, a), gl_canon(a)
    OP_MUL = 4,         // in: x(2) y(2)   out: gl_mul_fast(x0, y0), gl2_mul_fast(x, y) (2), fmul_any(x, y0) (2), gl2_mul(x, y) (2)
    OP_FOLD = 5,        // in: a0(2) a1(2) r(2) c(2) cr(2)
                        // out: fold(X a0, X a1, r) (2), fold(B a0.c0, B a1.c0, r) (2), fold_scaled(a0.c0, a1.c0, c, cr) (2)
    OP_LINE = 6,        // in: lo(2) hi(2) q0 q1 qinf
                        // out: slope(B), at_m1(B), slope(X) (2), at_m1(X) (2), q_at_m1(q0, q1, qinf)
    OP_CHAIN = 7,       // in: t_lo t_hi l_lo l_hi r_lo r_hi q0 q1
                        // out: the four grand-product fold sums of k_gp_fold (gp_kernels.cuh), the four of r0_accumulate (gp_fused.cuh)
    OP_FR = 8,          // in: a(4) b(4) raw Montgomery limbs   out: fr_add_dev, fr_sub_dev, fr_mul_dev32, fr_mul_dev (4 each)
    OP_FR_COND_SUB = 9, // in: t(5)   out: fr_cond_sub_dev (4)
    OP_FR_CANON = 10,   // in: x(4) canonical   out: fr_from_canonical(x) (4), fr_to_canonical(fr_from_canonical(x)) (4)
    OP_COUNT = 11
};

static const int kInWords[OP_COUNT] = {5, 9, 20, 2, 4, 10, 7, 8, 8, 5, 4};
static const int kOutWords[OP_COUNT] = {1, 1, 2, 3, 7, 6, 7, 8, 16, 4, 8};

__device__ __forceinline__ acc192 load_acc(const u64* p) {
    acc192 a;
    a.e01 = p[0]; a.e23 = p[1]; a.o01 = p[2]; a.e4 = (u32)p[3]; a.o2 = (u32)p[4];
    return a;
}
__device__ __forceinline__ fr load_fr(const u64* p) { return fr_make(p[0], p[1], p[2], p[3]); }
__device__ __forceinline__ void store_fr(u64* p, const fr& v) { p[0] = v.l[0]; p[1] = v.l[1]; p[2] = v.l[2]; p[3] = v.l[3]; }
__device__ __forceinline__ void store_x(u64* p, gl2 v) { p[0] = v.c0; p[1] = v.c1; }

__global__ void k_probe(int op, const u64* __restrict__ in, size_t in_words, size_t n, u64* __restrict__ out, size_t out_words) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const u64* a = in + i * in_words;
    u64* o = out + i * out_words;
    typedef GlField F;
    switch (op) {
    case OP_ACC_REDUCE: o[0] = acc_reduce(load_acc(a)); break;
    case OP_ACC_RUN: {
        acc192 s = load_acc(a);
        for (u64 k = 0; k < a[8]; k++) { acc_mad(s, a[5], a[6]); acc_add(s, a[7]); }
        o[0] = acc_reduce(s);
        break;
    }
    case OP_XACC: {
        xacc s;
        s.a00 = load_acc(a); s.a11 = load_acc(a + 5); s.ax = load_acc(a + 10);
        xacc_mad(s, gl2_make(a[15], a[16]), gl2_make(a[17], a[18]));
        xacc_mad_base(s, gl2_make(a[15], a[16]), a[19]);
        store_x(o, xacc_reduce(s));
        break;
    }
    case OP_SUB_ADD: o[0] = gl_sub_cs(a[0], a[1]); o[1] = gl_add_cs(a[1], a[0]); o[2] = gl_canon(a[0]); break;
    case OP_MUL: {
        const gl2 x = gl2_make(a[0], a[1]), y = gl2_make(a[2], a[3]);
        o[0] = gl_mul_fast(a[0], a[2]);
        store_x(o + 1, gl2_mul_fast(x, y));
        store_x(o + 3, F::fmul_any(x, a[2]));
        store_x(o + 5, gl2_mul(x, y));
        break;
    }
    case OP_FOLD: {
        const gl2 a0 = gl2_make(a[0], a[1]), a1 = gl2_make(a[2], a[3]), r = gl2_make(a[4], a[5]);
        const F::FoldAux aux = F::fold_aux(r);
        store_x(o, F::fold(a0, a1, r, aux));
        store_x(o + 2, F::fold(a[0], a[2], r, aux));
        store_x(o + 4, F::fold_scaled(a[0], a[2], gl2_make(a[6], a[7]), gl2_make(a[8], a[9])));
        break;
    }
    case OP_LINE: {
        const gl2 lo = gl2_make(a[0], a[1]), hi = gl2_make(a[2], a[3]);
        o[0] = F::slope(a[0], a[2]);
        o[1] = F::at_m1(a[0], a[2]);
        store_x(o + 2, F::slope(lo, hi));
        store_x(o + 4, F::at_m1(lo, hi));
        o[6] = F::q_at_m1(a[4], a[5], a[6]);
        break;
    }
    case OP_CHAIN: {
        const u64 t_lo = a[0], t_hi = a[1], l_lo = a[2], l_hi = a[3], r_lo = a[4], r_hi = a[5], q0 = a[6], q1 = a[7];
        F::BAcc s[4];
        for (int p = 0; p < 4; p++) s[p] = F::bacc_zero();
        // k_gp_fold: t sampled at 0, inf, -1, 1 times the product of the two children sampled at the same points
        F::bacc_mad(s[0], t_lo, F::fmul(l_lo, r_lo));
        F::bacc_mad(s[1], F::slope(t_lo, t_hi), F::fmul(F::slope(l_lo, l_hi), F::slope(r_lo, r_hi)));
        F::bacc_mad(s[2], F::at_m1(t_lo, t_hi), F::fmul(F::at_m1(l_lo, l_hi), F::at_m1(r_lo, r_hi)));
        F::bacc_mad(s[3], t_hi, F::fmul(l_hi, r_hi));
        for (int p = 0; p < 4; p++) o[p] = F::bacc_reduce(s[p]);
        // r0_accumulate
        F::BAcc d[4];
        for (int p = 0; p < 4; p++) d[p] = F::bacc_zero();
        const u64 qinf = F::fmul(F::slope(l_lo, l_hi), F::slope(r_lo, r_hi));
        const u64 qm1 = F::q_at_m1(q0, q1, qinf);
        F::bacc_mad(d[0], t_lo, q0);
        F::bacc_mad(d[1], F::slope(t_lo, t_hi), qinf);
        F::bacc_mad(d[2], F::at_m1(t_lo, t_hi), qm1);
        F::bacc_mad(d[3], t_hi, q1);
        for (int p = 0; p < 4; p++) o[4 + p] = F::bacc_reduce(d[p]);
        break;
    }
    case OP_FR: {
        const fr x = load_fr(a), y = load_fr(a + 4);
        store_fr(o, fr_add_dev(x, y));
        store_fr(o + 4, fr_sub_dev(x, y));
        store_fr(o + 8, fr_mul_dev32(x, y));
        store_fr(o + 12, fr_mul_dev(x, y));
        break;
    }
    case OP_FR_COND_SUB: store_fr(o, fr_cond_sub_dev(a[0], a[1], a[2], a[3], a[4])); break;
    case OP_FR_CANON: {
        const fr m = fr_from_canonical(a);
        store_fr(o, m);
        u64 c[4];
        fr_to_canonical(m, c);
        o[4] = c[0]; o[5] = c[1]; o[6] = c[2]; o[7] = c[3];
        break;
    }
    default: break;
    }
}

// Runs n_cases of `op` on the current device. Returns a cudaError_t (cudaErrorInvalidValue for an unknown op or a case row
// shorter than the op reads or writes).
extern "C" int probe_run(int op, const uint64_t* in, size_t in_words, size_t n_cases, uint64_t* out, size_t out_words) {
    if (op < 0 || op >= OP_COUNT || in_words < (size_t)kInWords[op] || out_words < (size_t)kOutWords[op]) return (int)cudaErrorInvalidValue;
    if (n_cases == 0) return 0;
    u64 *d_in = nullptr, *d_out = nullptr;
    cudaError_t e = cudaMalloc(&d_in, n_cases * in_words * sizeof(u64));
    if (e == cudaSuccess) e = cudaMalloc(&d_out, n_cases * out_words * sizeof(u64));
    if (e == cudaSuccess) e = cudaMemcpy(d_in, in, n_cases * in_words * sizeof(u64), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemset(d_out, 0, n_cases * out_words * sizeof(u64));
    if (e == cudaSuccess) {
        const unsigned threads = 128, blocks = (unsigned)((n_cases + threads - 1) / threads);
        k_probe<<<blocks, threads>>>(op, d_in, in_words, n_cases, d_out, out_words);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (e == cudaSuccess) e = cudaMemcpy(out, d_out, n_cases * out_words * sizeof(u64), cudaMemcpyDeviceToHost);
    cudaFree(d_in);
    cudaFree(d_out);
    return (int)e;
}
