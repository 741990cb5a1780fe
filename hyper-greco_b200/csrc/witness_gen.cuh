// Synthetic BFV secret-key-encryption witness on the device (SURVEY.md 8f item 4): the arithmetic of
// /root/reference/scripts/circuit_sk.py:72-140 (exact ct0i_hat = a_i s + e + k0_i k1 over Z, centred reduction mod
// (x^n + 1, q_i), r2i = (ct0i - ct0i_hat mod q_i) / (x^n + 1), r1i = (ct0i - ct0i_hat - r2i (x^n + 1)) / q_i, the bound
// assertions of :99-140) written straight into the input layout of BfvEncrypt::get_inputs
// (/root/reference/bfv-gkr/src/sk_encryption_circuit.rs:365-415; Poly::new_padded / new_shifted, poly.rs:21-44).
//
// The random draws (s ternary, e ~ N(0, 3.2^2) clipped, k1, a_i uniform; circuit_sk.py:29-70) stay with the caller: they are a few
// hundred kilobytes, and keeping them there makes the generator a pure function that the tests compare bit for bit with the numpy
// restatement (hyper-greco_b200/witness.py). What moves to the GPU is everything quadratic or per-coefficient in n:
//   k_wit_conv      exact negacyclic-free product a_i * s over Z, 128-bit accumulation, s in {-1, 0, 1}: (2n-1) n K integer MACs
//   k_wit_finish    per coefficient: + e + k0 k1, reduction by x^n + 1, centred mod q, quotients, bound checks, output layout
// Coefficients are lowest degree first inside the kernels; the outputs are highest degree first, negatives stored as p - |z|
// (circuit_sk.py:155-160), as canonical little-endian limbs of the field.
#pragma once
#include "prover.cuh"

namespace hg {

typedef __int128 i128;

struct WitGenStatus {  // all zero after a clean run
    unsigned not_multiple_of_cyclo;  // ct0i - ct0i_hat is not a multiple of x^n + 1 mod q (circuit_sk.py:116-118)
    unsigned not_multiple_of_q;      // the remainder is not divisible by q_i (:127-129)
    unsigned r1_out_of_range;        // :131-134
    unsigned r2_out_of_range;        // :119-122
};

// hat[i][k] = sum_j s[j] * a[i][k - j], k = 0 .. 2n-2 (lowest degree first). Tiles of 256 outputs x 1024 taps in shared memory.
constexpr int HG_WIT_KT = 256, HG_WIT_JT = 1024;
__global__ void __launch_bounds__(HG_WIT_KT) k_wit_conv(const signed char* __restrict__ s, const long long* __restrict__ a, int n, i128* __restrict__ hat) {
    __shared__ signed char ss[HG_WIT_JT];
    __shared__ long long sa[HG_WIT_JT + HG_WIT_KT];
    const int i = blockIdx.y, k0 = blockIdx.x * HG_WIT_KT, k = k0 + threadIdx.x;
    const long long* ai = a + (size_t)i * n;
    i128 acc = 0;
    for (int j0 = 0; j0 < n; j0 += HG_WIT_JT) {
        // taps j in [j0, j0 + JT), operands a[k - j] for k in [k0, k0 + KT): indices [k0 - j0 - JT + 1, k0 - j0 + KT)
        const int lo = k0 - j0 - HG_WIT_JT + 1;
        for (int t = threadIdx.x; t < HG_WIT_JT; t += HG_WIT_KT) ss[t] = j0 + t < n ? s[j0 + t] : 0;
        for (int t = threadIdx.x; t < HG_WIT_JT + HG_WIT_KT - 1; t += HG_WIT_KT) { const int idx = lo + t; sa[t] = (idx >= 0 && idx < n) ? ai[idx] : 0; }
        __syncthreads();
        // a[k - j] = sa[k - j - lo] = sa[threadIdx.x + JT - 1 - (j - j0)]
        long long part_lo = 0;  // |s a| < 2^59: 16 taps fit a 64-bit partial sum before it is widened
#pragma unroll 16
        for (int t = 0; t < HG_WIT_JT; t++) {
            part_lo += (long long)ss[t] * sa[threadIdx.x + HG_WIT_JT - 1 - t];
            if ((t & 15) == 15) { acc += (i128)part_lo; part_lo = 0; }
        }
        __syncthreads();
    }
    if (k < 2 * n - 1) hat[(size_t)i * (2 * n) + k] = acc;
}

__device__ __forceinline__ i128 wit_center(i128 x, long long q) {  // representative of x mod q in [-(q-1)/2, (q-1)/2]
    i128 r = x % (i128)q;
    if (r < 0) r += q;
    if (r > (i128)((q - 1) / 2)) r -= q;
    return r;
}
// canonical limbs of z mod p for |z| < 2^63: z >= 0 -> z, z < 0 -> p - |z|   (p given by its limbs, p > 2^63)
template <int LIMBS> __device__ __forceinline__ void wit_store(u64* dst, i128 z, const u64* p) {
    if (z >= 0) {
        dst[0] = (u64)z;
#pragma unroll
        for (int l = 1; l < LIMBS; l++) dst[l] = 0;
    } else {
        const u64 m = (u64)(-z);
        u64 borrow = 0;
#pragma unroll
        for (int l = 0; l < LIMBS; l++) {
            const u64 sub = l == 0 ? m : 0;
            const u64 d = p[l] - sub - borrow;
            borrow = (p[l] < sub + borrow || (sub + borrow < sub)) ? 1 : 0;
            dst[l] = d;
        }
    }
}
struct WitGenParams {
    int n, K;
    long long q[64], k0[64], r1_bound[64], r2_bound[64];
    u64 p[4];
};
// one thread per (modulus i, coefficient k < 2n): everything after the product, and the get_inputs layout.
// Outputs (LIMBS words per element, N2 = 2n):  ais [K][N2], r1is [K][N2], r2is [K][n], ct0is [K][N2]
template <int LIMBS>
__global__ void k_wit_finish(WitGenParams P, const signed char* __restrict__ e, const int* __restrict__ k1, const long long* __restrict__ a,
                             const i128* __restrict__ hat, u64* __restrict__ ais, u64* __restrict__ r1is, u64* __restrict__ r2is, u64* __restrict__ ct0is,
                             WitGenStatus* st) {
    const int n = P.n, N2 = 2 * n, i = blockIdx.y;
    const int k = blockIdx.x * blockDim.x + threadIdx.x;  // coefficient index, lowest degree first, 0 .. 2n-1
    if (k >= N2) return;
    const long long q = P.q[i];
    const i128* h = hat + (size_t)i * N2;
    auto hat_full = [&](int c) -> i128 {  // ct0i_hat coefficient c (degree c), c < 2n-1: a s + e + k0 k1 (the last two have degree < n)
        i128 v = h[c];
        if (c < n) v += (i128)e[c] + (i128)k1[c] * (i128)P.k0[i];
        return v;
    };
    // ---- ct0 (degree < n): (hat mod x^n + 1) centred mod q
    auto ct0_at = [&](int c) -> i128 {  // c < n
        i128 red = hat_full(c);
        if (c < n - 1) red -= hat_full(c + n);
        return wit_center(red, q);
    };
    // ---- num = ct0 - hat, centred mod q: its upper half is r2 (degree n-2 .. 0 <-> coefficients n .. 2n-2)
    auto numc_at = [&](int c) -> i128 {  // c < 2n-1
        i128 v = -hat_full(c);
        if (c < n) v += ct0_at(c);
        return wit_center(v, q);
    };
    u64* dst;
    if (k < n) {
        // ais: Poly::new_padded -> highest degree first, then n zeros
        dst = ais + ((size_t)i * N2 + (n - 1 - k)) * LIMBS;
        wit_store<LIMBS>(dst, (i128)a[(size_t)i * n + k], P.p);
        dst = ais + ((size_t)i * N2 + n + k) * LIMBS;
        wit_store<LIMBS>(dst, 0, P.p);
        // ct0is: new_shifted(ct0, 2n)[1:] + [0] -> n-1 zeros, the n coefficients highest degree first, one zero
        const i128 c0 = ct0_at(k);
        dst = ct0is + ((size_t)i * N2 + (n - 1) + (n - 1 - k)) * LIMBS;
        wit_store<LIMBS>(dst, c0, P.p);
        if (k < n - 1) { dst = ct0is + ((size_t)i * N2 + k) * LIMBS; wit_store<LIMBS>(dst, 0, P.p); }
        if (k == 0) { dst = ct0is + ((size_t)i * N2 + N2 - 1) * LIMBS; wit_store<LIMBS>(dst, 0, P.p); }
    }
    if (k == N2 - 1) {  // the padding element of r1is (2n-1 coefficients + one zero) and of r2is (n-1 coefficients + one zero)
        dst = r1is + ((size_t)i * N2 + N2 - 1) * LIMBS;
        wit_store<LIMBS>(dst, 0, P.p);
        dst = r2is + ((size_t)i * n + n - 1) * LIMBS;
        wit_store<LIMBS>(dst, 0, P.p);
        return;
    }
    // ---- r2 coefficient of degree d = k - n (k >= n), and the consistency checks of the lower half
    const i128 nc = numc_at(k);
    i128 r2_hi = 0, r2_lo = 0;  // r2 coefficients that touch rem[k]: rem[c] = num[c] - r2[c] (c < n-1) - r2[c - n] (c >= n)
    if (k >= n) {
        r2_hi = nc;  // r2[k - n]
        if ((r2_hi < 0 ? -r2_hi : r2_hi) > (i128)P.r2_bound[i]) atomicAdd(&st->r2_out_of_range, 1u);
        dst = r2is + ((size_t)i * n + (n - 2 - (k - n))) * LIMBS;   // n-1 coefficients, highest degree first
        wit_store<LIMBS>(dst, r2_hi, P.p);
    } else if (k < n - 1) {
        r2_lo = numc_at(k + n);  // r2[k]
        if (nc != r2_lo) atomicAdd(&st->not_multiple_of_cyclo, 1u);
    } else {  // k == n - 1
        if (nc != 0) atomicAdd(&st->not_multiple_of_cyclo, 1u);
    }
    // ---- r1 = (num - r2 (x^n + 1)) / q, all 2n-1 coefficients
    i128 rem = -hat_full(k);
    if (k < n) rem += ct0_at(k);
    rem -= (k >= n) ? r2_hi : r2_lo;
    if (rem % (i128)q != 0) atomicAdd(&st->not_multiple_of_q, 1u);
    const i128 r1 = rem / (i128)q;
    if ((r1 < 0 ? -r1 : r1) > (i128)P.r1_bound[i]) atomicAdd(&st->r1_out_of_range, 1u);
    dst = r1is + ((size_t)i * N2 + (N2 - 2 - k)) * LIMBS;  // 2n-1 coefficients highest degree first, then one zero
    wit_store<LIMBS>(dst, r1, P.p);
}
// s: new_padded -> [s high..low | n zeros];  e, k1: new_shifted(v, 2n - 1) -> [n-1 zeros | v high..low | one zero]
template <int LIMBS>
__global__ void k_wit_small(WitGenParams P, const signed char* __restrict__ s, const signed char* __restrict__ e, const int* __restrict__ k1,
                            u64* __restrict__ os, u64* __restrict__ oe, u64* __restrict__ ok1) {
    const int n = P.n, N2 = 2 * n;
    const int t = blockIdx.x * blockDim.x + threadIdx.x;  // output position
    if (t >= N2) return;
    i128 vs = 0, ve = 0, vk = 0;
    if (t < n) vs = s[n - 1 - t];
    if (t >= n - 1 && t < N2 - 1) { ve = e[n - 1 - (t - (n - 1))]; vk = k1[n - 1 - (t - (n - 1))]; }
    wit_store<LIMBS>(os + (size_t)t * LIMBS, vs, P.p);
    wit_store<LIMBS>(oe + (size_t)t * LIMBS, ve, P.p);
    wit_store<LIMBS>(ok1 + (size_t)t * LIMBS, vk, P.p);
}

// ---- BFV public-key encryption: the same arithmetic for two components per modulus,
//   ct0_i = pk0_i u + e0 + k0_i k1 + r1_i q_i + r2_i (x^n + 1)      ct1_i = pk1_i u + e1 + p1_i q_i + p2_i (x^n + 1)
//   k_wit_pk_conv    both exact products pk0_i * u and pk1_i * u over Z from one shared-memory tile of u: 2 (2n-1) n K integer MACs
//   k_wit_pk_finish  per (i, coefficient) and component: + e (+ k0 k1 for ct0), reduction by x^n + 1, centred mod q, quotients,
//                    bound checks, output layout
//   k_wit_pk_small   the layout of u, e0, e1, k1
struct WitGenPkStatus { WitGenStatus c[2]; };  // c[0]: ct0 (r1, r2), c[1]: ct1 (p1, p2)

// hat0[i][k] = sum_j u[j] pk0[i][k - j], hat1 likewise, k = 0 .. 2n-2 (lowest degree first)
__global__ void __launch_bounds__(HG_WIT_KT) k_wit_pk_conv(const signed char* __restrict__ u, const long long* __restrict__ pk0, const long long* __restrict__ pk1,
                                                          int n, i128* __restrict__ hat0, i128* __restrict__ hat1) {
    __shared__ signed char su[HG_WIT_JT];
    __shared__ long long s0[HG_WIT_JT + HG_WIT_KT], s1[HG_WIT_JT + HG_WIT_KT];
    const int i = blockIdx.y, k0 = blockIdx.x * HG_WIT_KT, k = k0 + threadIdx.x;
    const long long* a0 = pk0 + (size_t)i * n;
    const long long* a1 = pk1 + (size_t)i * n;
    i128 acc0 = 0, acc1 = 0;
    for (int j0 = 0; j0 < n; j0 += HG_WIT_JT) {
        const int lo = k0 - j0 - HG_WIT_JT + 1;
        for (int t = threadIdx.x; t < HG_WIT_JT; t += HG_WIT_KT) su[t] = j0 + t < n ? u[j0 + t] : 0;
        for (int t = threadIdx.x; t < HG_WIT_JT + HG_WIT_KT - 1; t += HG_WIT_KT) {
            const int idx = lo + t;
            const bool in = idx >= 0 && idx < n;
            s0[t] = in ? a0[idx] : 0;
            s1[t] = in ? a1[idx] : 0;
        }
        __syncthreads();
        long long part0 = 0, part1 = 0;  // |u pk| < 2^59 (checked by the caller): 16 taps fit a 64-bit partial sum before it is widened
#pragma unroll 16
        for (int t = 0; t < HG_WIT_JT; t++) {
            const long long uv = su[t];
            part0 += uv * s0[threadIdx.x + HG_WIT_JT - 1 - t];
            part1 += uv * s1[threadIdx.x + HG_WIT_JT - 1 - t];
            if ((t & 15) == 15) { acc0 += (i128)part0; acc1 += (i128)part1; part0 = 0; part1 = 0; }
        }
        __syncthreads();
    }
    if (k < 2 * n - 1) { hat0[(size_t)i * (2 * n) + k] = acc0; hat1[(size_t)i * (2 * n) + k] = acc1; }
}

struct WitGenPkParams {
    int n, K;
    long long q[64], k0[64], q1_bound[2][64], q2_bound[2][64];  // [component][i]: r1 / p1 and r2 / p2 bounds
    u64 p[4];
};
// One component of one (modulus i, coefficient k < 2n): ct = (hat mod x^n + 1) centred mod q, q2 = the upper half of (ct - hat) centred,
// q1 = (ct - hat - q2 (x^n + 1)) / q. `extra(c)` is the part of hat of degree < n added to the product (e, and k0 k1 for ct0).
// Outputs: pk [N2] (padded), q1 [N2], q2 [n], ct [N2], in the layouts of k_wit_finish.
template <int LIMBS, class Extra>
__device__ __forceinline__ void wit_pk_component(const WitGenPkParams& P, int i, int k, const long long* __restrict__ pk, const i128* __restrict__ h, Extra extra,
                                                 u64* __restrict__ opk, u64* __restrict__ oq1, u64* __restrict__ oq2, u64* __restrict__ oct,
                                                 long long q1_bound, long long q2_bound, WitGenStatus* st) {
    const int n = P.n, N2 = 2 * n;
    const long long q = P.q[i];
    auto hat_full = [&](int c) -> i128 { i128 v = h[c]; if (c < n) v += extra(c); return v; };
    auto ct_at = [&](int c) -> i128 {
        i128 red = hat_full(c);
        if (c < n - 1) red -= hat_full(c + n);
        return wit_center(red, q);
    };
    auto numc_at = [&](int c) -> i128 {
        i128 v = -hat_full(c);
        if (c < n) v += ct_at(c);
        return wit_center(v, q);
    };
    if (k < n) {
        wit_store<LIMBS>(opk + (size_t)(n - 1 - k) * LIMBS, (i128)pk[k], P.p);
        wit_store<LIMBS>(opk + (size_t)(n + k) * LIMBS, 0, P.p);
        wit_store<LIMBS>(oct + (size_t)((n - 1) + (n - 1 - k)) * LIMBS, ct_at(k), P.p);
        if (k < n - 1) wit_store<LIMBS>(oct + (size_t)k * LIMBS, 0, P.p);
        if (k == 0) wit_store<LIMBS>(oct + (size_t)(N2 - 1) * LIMBS, 0, P.p);
    }
    if (k == N2 - 1) {
        wit_store<LIMBS>(oq1 + (size_t)(N2 - 1) * LIMBS, 0, P.p);
        wit_store<LIMBS>(oq2 + (size_t)(n - 1) * LIMBS, 0, P.p);
        return;
    }
    const i128 nc = numc_at(k);
    i128 q2_hi = 0, q2_lo = 0;
    if (k >= n) {
        q2_hi = nc;
        if ((q2_hi < 0 ? -q2_hi : q2_hi) > (i128)q2_bound) atomicAdd(&st->r2_out_of_range, 1u);
        wit_store<LIMBS>(oq2 + (size_t)(n - 2 - (k - n)) * LIMBS, q2_hi, P.p);
    } else if (k < n - 1) {
        q2_lo = numc_at(k + n);
        if (nc != q2_lo) atomicAdd(&st->not_multiple_of_cyclo, 1u);
    } else {
        if (nc != 0) atomicAdd(&st->not_multiple_of_cyclo, 1u);
    }
    i128 rem = -hat_full(k);
    if (k < n) rem += ct_at(k);
    rem -= (k >= n) ? q2_hi : q2_lo;
    if (rem % (i128)q != 0) atomicAdd(&st->not_multiple_of_q, 1u);
    const i128 q1 = rem / (i128)q;
    if ((q1 < 0 ? -q1 : q1) > (i128)q1_bound) atomicAdd(&st->r1_out_of_range, 1u);
    wit_store<LIMBS>(oq1 + (size_t)(N2 - 2 - k) * LIMBS, q1, P.p);
}
// one thread per (modulus i, coefficient k < 2n), both components. Outputs (LIMBS words per element, N2 = 2n):
//   pk0is, pk1is, r1is, p1is, ct0is, ct1is [K][N2];  r2is, p2is [K][n]
template <int LIMBS>
__global__ void k_wit_pk_finish(WitGenPkParams P, const signed char* __restrict__ e0, const signed char* __restrict__ e1, const int* __restrict__ k1,
                                const long long* __restrict__ pk0, const long long* __restrict__ pk1, const i128* __restrict__ hat0, const i128* __restrict__ hat1,
                                u64* __restrict__ pk0is, u64* __restrict__ pk1is, u64* __restrict__ r1is, u64* __restrict__ p1is, u64* __restrict__ r2is,
                                u64* __restrict__ p2is, u64* __restrict__ ct0is, u64* __restrict__ ct1is, WitGenPkStatus* st) {
    const int n = P.n, N2 = 2 * n, i = blockIdx.y;
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= N2) return;
    const size_t wide = (size_t)i * N2 * LIMBS, narrow = (size_t)i * n * LIMBS;
    const long long k0 = P.k0[i];
    wit_pk_component<LIMBS>(P, i, k, pk0 + (size_t)i * n, hat0 + (size_t)i * N2, [&](int c) { return (i128)e0[c] + (i128)k1[c] * (i128)k0; },
                            pk0is + wide, r1is + wide, r2is + narrow, ct0is + wide, P.q1_bound[0][i], P.q2_bound[0][i], &st->c[0]);
    wit_pk_component<LIMBS>(P, i, k, pk1 + (size_t)i * n, hat1 + (size_t)i * N2, [&](int c) { return (i128)e1[c]; },
                            pk1is + wide, p1is + wide, p2is + narrow, ct1is + wide, P.q1_bound[1][i], P.q2_bound[1][i], &st->c[1]);
}
// u: new_padded -> [u high..low | n zeros];  e0, e1, k1: new_shifted(v, 2n - 1) -> [n-1 zeros | v high..low | one zero]
template <int LIMBS>
__global__ void k_wit_pk_small(WitGenPkParams P, const signed char* __restrict__ u, const signed char* __restrict__ e0, const signed char* __restrict__ e1,
                               const int* __restrict__ k1, u64* __restrict__ ou, u64* __restrict__ oe0, u64* __restrict__ oe1, u64* __restrict__ ok1) {
    const int n = P.n, N2 = 2 * n;
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= N2) return;
    i128 vu = 0, v0 = 0, v1 = 0, vk = 0;
    if (t < n) vu = u[n - 1 - t];
    if (t >= n - 1 && t < N2 - 1) { const int c = n - 1 - (t - (n - 1)); v0 = e0[c]; v1 = e1[c]; vk = k1[c]; }
    wit_store<LIMBS>(ou + (size_t)t * LIMBS, vu, P.p);
    wit_store<LIMBS>(oe0 + (size_t)t * LIMBS, v0, P.p);
    wit_store<LIMBS>(oe1 + (size_t)t * LIMBS, v1, P.p);
    wit_store<LIMBS>(ok1 + (size_t)t * LIMBS, vk, P.p);
}

}  // namespace hg
