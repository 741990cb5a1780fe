// Grand-product layer sumcheck kernels (K8; /root/reference/lasso/src/memory_checking/prover.rs:223-279), the dominant
// cost of the Lasso node. One round of
//        g = t_0 * sum_i c_i * l_i * r_i          (t_0 = l_0, F4/Q2; c_i = gamma^i under A5)
// per launch, evaluation fused with the fold by the previous challenge.
//   * work is split over (pair-index tiles) x (term groups) so that small rounds still fill the GPU and every thread has
//     several independent 256-bit loads in flight;
//   * h(X) = sum_i c_i sum_b t_0 l_i r_i is linear in the terms, so the c_i are folded into the TABLES once (round 1
//     writes l'_i = c_i * l_i; folding is linear, later rounds never multiply by c_i again) and the final evaluations are
//     unscaled on the host with c_i^{-1}. Field arithmetic is exact, so the messages are bit-identical;
//   * the round polynomial is sampled at X = 0, infinity (leading coefficient) and -1: those line values cost one
//     subtraction each. Together with the running TRUE sum h(0) + h(1) (tracked on the host, h(1) is sampled only in
//     round 0) they determine the cubic exactly; the host derives whatever the wire format needs (A3);
//   * products are accumulated unreduced (gl.cuh acc192 / xacc) and reduced once per accumulator: the kernels are bound by
//     the integer ALU pipe, not by HBM, so instruction count is what matters (profiles/).
// Message slots: [h(0), h(inf), h(-1)] and, in round 0 only, [.., h(1)].
#pragma once
#include "bn254.cuh"
#include "kernels.cuh"

namespace hg {

// ---- 256-bit global loads / stores (LDG.E.256 / STG.E.256 on sm_100a), streaming (no L1 allocation)
__device__ __forceinline__ void ldg256(const void* p, u64& a, u64& b, u64& c, u64& d) {
    asm volatile("ld.global.nc.L1::no_allocate.v4.u64 {%0,%1,%2,%3}, [%4];" : "=l"(a), "=l"(b), "=l"(c), "=l"(d) : "l"(p));
}
__device__ __forceinline__ void stg256(void* p, u64 a, u64 b, u64 c, u64 d) {
    asm volatile("st.global.L1::no_allocate.v4.u64 [%0], {%1,%2,%3,%4};" ::"l"(p), "l"(a), "l"(b), "l"(c), "l"(d) : "memory");
}
__device__ __forceinline__ void ldg128(const void* p, u64& a, u64& b) {
    asm volatile("ld.global.nc.L1::no_allocate.v2.u64 {%0,%1}, [%2];" : "=l"(a), "=l"(b) : "l"(p));
}
// four consecutive elements starting at p (32-byte aligned)
__device__ __forceinline__ void load4(const u64* p, u64 (&v)[4]) { ldg256(p, v[0], v[1], v[2], v[3]); }
__device__ __forceinline__ void load4(const gl2* p, gl2 (&v)[4]) {
    ldg256(p, v[0].c0, v[0].c1, v[1].c0, v[1].c1);
    ldg256(p + 2, v[2].c0, v[2].c1, v[3].c0, v[3].c1);
}
__device__ __forceinline__ void load2(const u64* p, u64 (&v)[2]) { ldg128(p, v[0], v[1]); }
__device__ __forceinline__ void load2(const gl2* p, gl2 (&v)[2]) { ldg256(p, v[0].c0, v[0].c1, v[1].c0, v[1].c1); }
__device__ __forceinline__ void store2(gl2* p, gl2 a, gl2 b) { stg256(p, a.c0, a.c1, b.c0, b.c1); }
__device__ __forceinline__ void store1(gl2* p, gl2 a) {
    asm volatile("st.global.L1::no_allocate.v2.u64 [%0], {%1,%2};" ::"l"(p), "l"(a.c0), "l"(a.c1) : "memory");
}
// BN254: one element = one 256-bit access
__device__ __forceinline__ void load4(const fr* p, fr (&v)[4]) {
#pragma unroll
    for (int i = 0; i < 4; i++) ldg256(p + i, v[i].l[0], v[i].l[1], v[i].l[2], v[i].l[3]);
}
__device__ __forceinline__ void load2(const fr* p, fr (&v)[2]) {
    ldg256(p, v[0].l[0], v[0].l[1], v[0].l[2], v[0].l[3]);
    ldg256(p + 1, v[1].l[0], v[1].l[1], v[1].l[2], v[1].l[3]);
}
__device__ __forceinline__ void store2(fr* p, fr a, fr b) {
    stg256(p, a.l[0], a.l[1], a.l[2], a.l[3]);
    stg256(p + 1, b.l[0], b.l[1], b.l[2], b.l[3]);
}
__device__ __forceinline__ void store1(fr* p, fr a) { stg256(p, a.l[0], a.l[1], a.l[2], a.l[3]); }
// pull the bytes a later iteration will load into L2 (costs no registers; the loop is otherwise latency-bound, profiles/)
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

// ---- round 0: base-field tables [nvec][2n] (l_i = first half, r_i = second half of vector i), n = 2^nv
//      msg: h(0), h(inf), h(-1), h(1)
template <class FP, int U>
__global__ void __launch_bounds__(HG_BLOCK)
k_gp_r0(const typename FP::B* __restrict__ tables, size_t n, int nvec, int tpg, const typename FP::X* __restrict__ coeffs,
        typename FP::X* partials, unsigned* counter, typename FP::X* msg) {
    typedef typename FP::B B;
    typedef typename FP::X X;
    constexpr int NP = 4;
    const size_t npairs = n / 2, stride = (size_t)gridDim.x * blockDim.x;
    const int i0 = blockIdx.y * tpg, i1 = min(nvec, i0 + tpg);
    typename FP::XAcc accx[NP];
#pragma unroll
    for (int p = 0; p < NP; p++) accx[p] = FP::xacc_zero_();
    for (size_t b0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x; b0 < npairs; b0 += stride * U) {
        B t0[U][NP];
#pragma unroll
        for (int u = 0; u < U; u++) {
            const size_t b = b0 + u * stride;
            B p[2] = {FP::b_zero(), FP::b_zero()};
            if (b < npairs) load2(tables + 2 * b, p);
            t0[u][0] = p[0]; t0[u][1] = FP::slope(p[0], p[1]); t0[u][2] = FP::at_m1(p[0], p[1]); t0[u][3] = p[1];
        }
        for (int i = i0; i < i1; i++) {
            const B* li = tables + (size_t)i * 2 * n;
            const B* ri = li + n;
            B l[U][2], r[U][2];
#pragma unroll
            for (int u = 0; u < U; u++) {
                const size_t b = b0 + u * stride;
                l[u][0] = l[u][1] = r[u][0] = r[u][1] = FP::b_zero();
                if (b < npairs) { load2(li + 2 * b, l[u]); load2(ri + 2 * b, r[u]); }
            }
            typename FP::BAcc s[NP];
#pragma unroll
            for (int p = 0; p < NP; p++) s[p] = FP::bacc_zero();
#pragma unroll
            for (int u = 0; u < U; u++) {
                FP::bacc_mad(s[0], t0[u][0], FP::fmul(l[u][0], r[u][0]));
                FP::bacc_mad(s[1], t0[u][1], FP::fmul(FP::slope(l[u][0], l[u][1]), FP::slope(r[u][0], r[u][1])));
                FP::bacc_mad(s[2], t0[u][2], FP::fmul(FP::at_m1(l[u][0], l[u][1]), FP::at_m1(r[u][0], r[u][1])));
                FP::bacc_mad(s[3], t0[u][3], FP::fmul(l[u][1], r[u][1]));
            }
            const X c = coeffs[i];
#pragma unroll
            for (int p = 0; p < NP; p++) FP::xacc_mad_b(accx[p], c, FP::bacc_reduce(s[p]));
        }
    }
    X acc[NP];
#pragma unroll
    for (int p = 0; p < NP; p++) acc[p] = FP::xacc_reduce_(accx[p]);
    block_reduce_finalize<FP, NP, true>(acc, partials, counter, msg);
}

// ---- rounds >= 1: fold by r_prev, write the folded tables, evaluate the next round polynomial on them
//   in : [2*nvec][n_in] (TIN = B in round 1, X later);  out: [2*nvec][n_in/2]
//   SCALE (round 1, TIN = B): l_i (i > 0) is written as c_i * l_i and r_0 as c_0 * r_0 (l_0 stays: it is also t_0);
//   cr[i] = c_i * r_prev is precomputed (k_gp_coeffs)
//   msg: h(0), h(inf), h(-1)
template <class FP, class TIN, bool SCALE>
__global__ void __launch_bounds__(HG_BLOCK)
k_gp_fold(const TIN* __restrict__ in, typename FP::X* __restrict__ out, size_t n_in, int nvec, int tpg,
          const typename FP::X* __restrict__ coeffs, const typename FP::X* __restrict__ cr, const typename FP::X* __restrict__ r_prev,
          typename FP::X* partials, unsigned* counter, typename FP::X* msg) {
    typedef typename FP::X X;
    constexpr int NP = 3;
    const size_t npairs = n_in / 4, n_out = n_in / 2;
    const int i0 = blockIdx.y * tpg, i1 = min(nvec, i0 + tpg);
    const X r = *r_prev;
    const typename FP::FoldAux aux = FP::fold_aux(r);
    X acc[NP];
#pragma unroll
    for (int p = 0; p < NP; p++) acc[p] = FP::x_zero();
    for (size_t b = (size_t)blockIdx.x * blockDim.x + threadIdx.x; b < npairs; b += (size_t)gridDim.x * blockDim.x) {
        X t0[NP];
        {
            TIN a[4];
            load4(in + 4 * b, a);
            X lo = FP::fold(a[0], a[1], r, aux), hi = FP::fold(a[2], a[3], r, aux);
            t0[0] = lo; t0[1] = FP::slope(lo, hi); t0[2] = FP::at_m1(lo, hi);
        }
        typename FP::XAcc P[NP];
#pragma unroll
        for (int p = 0; p < NP; p++) P[p] = FP::xacc_zero_();
        for (int i = i0; i < i1; i++) {
            TIN a[4], c[4];
            load4(in + (size_t)(2 * i) * n_in + 4 * b, a);
            load4(in + (size_t)(2 * i + 1) * n_in + 4 * b, c);
            X l_lo, l_hi, r_lo, r_hi;
            if constexpr (SCALE) {
                // term i carries c_i on l_i; term 0 carries c_0 on r_0, because l_0 is also the common factor t_0
                const X ci = coeffs[i], cri = cr[i];
                if (i > 0) {
                    l_lo = FP::fold_scaled(a[0], a[1], ci, cri); l_hi = FP::fold_scaled(a[2], a[3], ci, cri);
                    r_lo = FP::fold(c[0], c[1], r, aux); r_hi = FP::fold(c[2], c[3], r, aux);
                } else {
                    l_lo = FP::fold(a[0], a[1], r, aux); l_hi = FP::fold(a[2], a[3], r, aux);
                    r_lo = FP::fold_scaled(c[0], c[1], ci, cri); r_hi = FP::fold_scaled(c[2], c[3], ci, cri);
                }
            } else {
                l_lo = FP::fold(a[0], a[1], r, aux); l_hi = FP::fold(a[2], a[3], r, aux);
                r_lo = FP::fold(c[0], c[1], r, aux); r_hi = FP::fold(c[2], c[3], r, aux);
            }
            store2(out + (size_t)(2 * i) * n_out + 2 * b, l_lo, l_hi);
            store2(out + (size_t)(2 * i + 1) * n_out + 2 * b, r_lo, r_hi);
            FP::xacc_mad_(P[0], l_lo, r_lo);
            FP::xacc_mad_(P[1], FP::slope(l_lo, l_hi), FP::slope(r_lo, r_hi));
            FP::xacc_mad_(P[2], FP::at_m1(l_lo, l_hi), FP::at_m1(r_lo, r_hi));
        }
#pragma unroll
        for (int p = 0; p < NP; p++) acc[p] = FP::x_add(acc[p], FP::fmul(t0[p], FP::xacc_reduce_(P[p])));
    }
    block_reduce_finalize<FP, NP, true>(acc, partials, counter, msg);
}

// per-layer coefficient tables: c[i] = gamma^i (A5: or reversed), cr[i] = c[i] * r_0 when r0 != nullptr
template <class FP>
__global__ void k_gp_coeffs(const typename FP::X* __restrict__ gamma, const typename FP::X* __restrict__ r0, int n, int ascending,
                            typename FP::X* __restrict__ c, typename FP::X* __restrict__ cr) {
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    typename FP::X p = FP::x_one(), g = *gamma;
    for (int i = 0; i < n; i++) {
        const int k = ascending ? i : n - 1 - i;
        c[k] = p;
        if (r0) cr[k] = FP::x_mul(p, *r0);
        p = FP::x_mul(p, g);
    }
}

}  // namespace hg

// =========================================================================================================
// Batched (prefetch-mode) variants. With the challenges known up front every layer of both grand products is an
// independent sumcheck, so round j of ALL layers runs in ONE launch (a grid partitioned by a descriptor table), and the
// last rounds of every layer (tables of <= HG_GP_TAIL elements) run in ONE launch with one CTA per layer, tables in
// shared memory. ~430 launches per proof become ~20.
namespace hg {

// table length at which a layer moves to the shared-memory tail kernel: FP::GP_TAIL_LOG (64 elements of 16 B for
// Goldilocks, 32 elements of 32 B for BN254: 2*m tables * 1.5 * that must fit 227 KB)
constexpr int HG_TAIL_THREADS = 256;
constexpr int HG_GP_TAIL_MAXR = 10;  // most rounds the tail kernel runs (tables of up to 2^11 entries)
// threads per CTA of the batched streaming kernels: FP::GP_BLOCK (128 for Goldilocks: same registers per thread, twice the CTAs
// per SM, 3 % faster; 256 for BN254)
#ifndef HG_GP_PREFETCH
#define HG_GP_PREFETCH 1
#endif

template <class FP> struct GpItem {
    const void* in;                  // tables read this round (base in round 1, extension later): [2*nvec][n_in]
    typename FP::X* out;             // tables written this round (see k_gp_fold_multi)
    unsigned long long n_in;
    const typename FP::X* c;         // c_i
    const typename FP::X* cr;        // c_i * r_0 (round 1)
    const typename FP::X* r_prev;    // challenge of the previous round, folded on read (round 1)
    const typename FP::X* r_cur;     // challenge of this round, folded on write
    typename FP::X* msg;
    typename FP::X* partials;
    unsigned* counter;
    int nvec, tpg, bx, groups;
    int blk_start, nblk;
    int i_begin, i_end;              // terms (vectors) this device owns: a proof can be split over GPUs by terms (h is linear in them)
    int write_t0;                    // table 0 (= t_0) is folded by every device; written here when term 0 is not owned
};

template <class FP, int NP>
__device__ __forceinline__ void block_reduce_finalize_ex(typename FP::X (&acc)[NP], typename FP::X* partials, unsigned* counter,
                                                         typename FP::X* out, unsigned nblk, unsigned bid) {
    typedef typename FP::X X;
    __shared__ X sm[32][NP];
    __shared__ bool is_last;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = (blockDim.x + 31) >> 5;
#pragma unroll
    for (int p = 0; p < NP; p++) {
        X v = acc[p];
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) v = FP::x_add(v, FP::x_shfl_down(v, off));
        if (lane == 0) sm[warp][p] = v;
    }
    __syncthreads();
    if (warp == 0) {
#pragma unroll
        for (int p = 0; p < NP; p++) {
            X v = lane < nwarps ? sm[lane][p] : FP::x_zero();
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) v = FP::x_add(v, FP::x_shfl_down(v, off));
            if (lane == 0) partials[(size_t)bid * NP + p] = v;
        }
    }
    if (threadIdx.x == 0) {
        __threadfence();
        unsigned t = atomicAdd(counter, 1u);
        is_last = (t == nblk - 1);
    }
    __syncthreads();
    if (!is_last) return;
    __threadfence();
    X s[NP];
#pragma unroll
    for (int p = 0; p < NP; p++) s[p] = FP::x_zero();
    for (unsigned b = threadIdx.x; b < nblk; b += blockDim.x)
#pragma unroll
        for (int p = 0; p < NP; p++) s[p] = FP::x_add(s[p], FP::x_ldcg(partials + (size_t)b * NP + p));
    __syncthreads();
#pragma unroll
    for (int p = 0; p < NP; p++) {
        X v = s[p];
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) v = FP::x_add(v, FP::x_shfl_down(v, off));
        if (lane == 0) sm[warp][p] = v;
    }
    __syncthreads();
    if (warp == 0) {
#pragma unroll
        for (int p = 0; p < NP; p++) {
            X v = lane < nwarps ? sm[lane][p] : FP::x_zero();
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) v = FP::x_add(v, FP::x_shfl_down(v, off));
            if (lane == 0) out[p] = v;
        }
        if (lane == 0) *counter = 0;
    }
}

// which item does this block belong to: largest k with items[k].blk_start <= blockIdx.x (binary search over <= ~70 items)
template <class ITEM> __device__ __forceinline__ int find_item(const ITEM* items, int nitems) {
    int lo = 0, hi = nitems - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if ((int)blockIdx.x >= items[mid].blk_start) lo = mid; else hi = mid - 1;
    }
    return lo;
}
template <class FP> __device__ __forceinline__ int gp_find_item(const GpItem<FP>* items, int nitems) { return find_item(items, nitems); }

// Round r (>= 1) of a layer sumcheck samples h_r on the pairs (2b, 2b+1) of the level-r tables L_r and writes every pair folded
// by its own challenge r_cur, i.e. L_{r+1}: all challenges are on the device before the launch, so the next round reads half as
// much and folds nothing on read.
//   SCALE (round 1, TIN = B): reads quads of the base tables L_0 and folds them by r_prev = r_0 into the pairs of L_1, scaling
//     them as it goes; l_i (i > 0) is written as c_i * l_i and r_0 as c_0 * r_0 (l_0 stays: it is also t_0).
//   otherwise (TIN = X): reads the pairs of L_r as the previous round wrote them.
//   in: [2*nvec][n_in] (n_in = |L_0| or |L_r|);  out: [2*nvec][n_in / 4 or n_in / 2] (|L_{r+1}|)
template <class FP, class TIN, bool SCALE>
__global__ void __launch_bounds__(FP::GP_BLOCK, FP::GP_FOLD_CTAS) k_gp_fold_multi(const GpItem<FP>* __restrict__ items, int nitems) {
    typedef typename FP::X X;
    constexpr bool QUAD = SCALE;
    constexpr int NP = 3, W = QUAD ? 4 : 2;  // W: entries of a table read per position
    const GpItem<FP> it = items[gp_find_item<FP>(items, nitems)];
    const unsigned lb = blockIdx.x - it.blk_start;
    const unsigned bxi = lb % it.bx, grp = lb / it.bx;
    const TIN* in = (const TIN*)it.in;
    X* out = it.out;
    const size_t n_in = it.n_in, npairs = n_in / W, n_out = npairs;
    const int i0 = it.i_begin + grp * it.tpg, i1 = min(it.i_end, i0 + it.tpg);
    X r = FP::x_zero();
    if constexpr (QUAD) r = *it.r_prev;
    const X rc = *it.r_cur;
    const typename FP::FoldAux aux = FP::fold_aux(r), auxc = FP::fold_aux(rc);
    // one pair of L_r: folded from its quad of L_{r-1}, or as read
    auto pair = [&](const TIN (&a)[W], X& lo, X& hi) {
        if constexpr (QUAD) { lo = FP::fold(a[0], a[1], r, aux); hi = FP::fold(a[2], a[3], r, aux); }
        else { lo = a[0]; hi = a[1]; }
    };
    auto load = [&](const TIN* p, TIN (&a)[W]) {
        if constexpr (QUAD) load4(p, a); else load2(p, a);
    };
    auto store = [&](X* tab, size_t b, X lo, X hi) { store1(tab + b, FP::fold(lo, hi, rc, auxc)); };
    X acc[NP];
#pragma unroll
    for (int p = 0; p < NP; p++) acc[p] = FP::x_zero();
    for (size_t b = (size_t)bxi * blockDim.x + threadIdx.x; b < npairs; b += (size_t)it.bx * blockDim.x) {
        X t0[NP];
        {
            TIN a[W];
            load(in + W * b, a);
            X lo, hi;
            pair(a, lo, hi);
            t0[0] = lo; t0[1] = FP::slope(lo, hi); t0[2] = FP::at_m1(lo, hi);
            if (it.write_t0 && grp == 0) store(out, b, lo, hi);
        }
        typename FP::XAcc P[NP];
#pragma unroll
        for (int p = 0; p < NP; p++) P[p] = FP::xacc_zero_();
        for (int i = i0; i < i1; i++) {
            TIN a[W], c[W];
            load(in + (size_t)(2 * i) * n_in + W * b, a);
            load(in + (size_t)(2 * i + 1) * n_in + W * b, c);
            if (i + HG_GP_PREFETCH < i1) {
                prefetch_l2(in + (size_t)(2 * (i + HG_GP_PREFETCH)) * n_in + W * b);
                prefetch_l2(in + (size_t)(2 * (i + HG_GP_PREFETCH) + 1) * n_in + W * b);
            }
            X l_lo, l_hi, r_lo, r_hi;
            if constexpr (SCALE) {
                // term i carries c_i on l_i; term 0 carries c_0 on r_0, because l_0 is also the common factor t_0
                const X ci = it.c[i], cri = it.cr[i];
                if (i > 0) {
                    l_lo = FP::fold_scaled(a[0], a[1], ci, cri); l_hi = FP::fold_scaled(a[2], a[3], ci, cri);
                    pair(c, r_lo, r_hi);
                } else {
                    pair(a, l_lo, l_hi);
                    r_lo = FP::fold_scaled(c[0], c[1], ci, cri); r_hi = FP::fold_scaled(c[2], c[3], ci, cri);
                }
            } else {
                pair(a, l_lo, l_hi);
                pair(c, r_lo, r_hi);
            }
            store(out + (size_t)(2 * i) * n_out, b, l_lo, l_hi);
            store(out + (size_t)(2 * i + 1) * n_out, b, r_lo, r_hi);
            // q_i(X) = l_i(X) r_i(X) is quadratic: sampled at X = 0, 1, inf (no value at -1 inside the term loop)
            FP::xacc_mad_(P[0], l_lo, r_lo);
            FP::xacc_mad_(P[1], FP::slope(l_lo, l_hi), FP::slope(r_lo, r_hi));
            FP::xacc_mad_(P[2], l_hi, r_hi);
        }
        // Q(-1) = 2 Q(0) - Q(1) + 2 Q(inf) for the summed quadratic Q = sum_i q_i; h sampled at 0, inf, -1 as before
        const X Q0 = FP::xacc_reduce_(P[0]), Qi = FP::xacc_reduce_(P[1]), Q1 = FP::xacc_reduce_(P[2]);
        const X Qs = FP::x_add(Q0, Qi), Qm = FP::x_sub(FP::x_add(Qs, Qs), Q1);
        acc[0] = FP::x_add(acc[0], FP::fmul(t0[0], Q0));
        acc[1] = FP::x_add(acc[1], FP::fmul(t0[1], Qi));
        acc[2] = FP::x_add(acc[2], FP::fmul(t0[2], Qm));
    }
    block_reduce_finalize_ex<FP, NP>(acc, it.partials, it.counter, it.msg, it.nblk, lb);
}

// coefficient tables of all layers in one launch: block = layer
template <class FP> struct GpCoeffItem {
    const typename FP::X* gamma;
    const typename FP::X* r0;  // may be nullptr (layers with a single round)
    typename FP::X* c;
    typename FP::X* cr;
    int n;
};
template <class FP> __global__ void k_gp_coeffs_multi(const GpCoeffItem<FP>* __restrict__ items, int ascending) {
    const GpCoeffItem<FP> it = items[blockIdx.x];
    const typename FP::X g = *it.gamma;
    // thread i: gamma^i by square and multiply (a serial chain of n products took 23 us on the critical path)
    for (int i = threadIdx.x; i < it.n; i += blockDim.x) {
        typename FP::X p = FP::x_one(), b = g;
        for (int e = i; e; e >>= 1) { if (e & 1) p = FP::x_mul(p, b); b = FP::x_mul(b, b); }
        const int k = ascending ? i : it.n - 1 - i;
        it.c[k] = p;
        if (it.r0) it.cr[k] = FP::x_mul(p, *it.r0);
    }
}

// ---- tail: one CTA per layer, tables in shared memory, all remaining rounds + the final evaluations
template <class FP> struct GpTailItem {
    const void* in;                 // from_base: base tables [nvec][2n]; else extension tables [2*nvec][n] (already scaled)
    const typename FP::X* c;
    const typename FP::X* chal;     // chal[k] = challenge folded in the k-th folding tail round; chal[rounds] = last challenge (final fold)
    typename FP::X* msg0;           // from_base: 4 slots for round 0
    typename FP::X* msg;            // 3 slots per sampled tail round (!from_base: `rounds` + 1 of them, see k_gp_tail)
    typename FP::X* evals;          // 2*nvec final evaluations (l_i for i > 0 scaled by c_i, r_0 by c_0)
    int from_base, n, nvec, rounds;
    int i_begin, i_end;             // owned terms (see GpItem)
    const typename FP::X* r0part;   // !from_base: round-0 partial sums of the fused tree builders (gp_fused.cuh), [r0n][4], summed into msg0
    int r0n;
    // the layer's terms are split over `groups` CTAs of tpg terms; gpart: [groups][1 + HG_GP_TAIL_MAXR][4] partial sums
    int tpg, groups;
    typename FP::X* gpart;
    unsigned* counter;
};

template <class FP, int NP>
__device__ __forceinline__ void tail_block_sum(typename FP::X (&acc)[NP], typename FP::X* red /*[32][NP]*/, typename FP::X* out) {
    typedef typename FP::X X;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
#pragma unroll
    for (int p = 0; p < NP; p++) {
        X v = acc[p];
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) v = FP::x_add(v, FP::x_shfl_down(v, off));
        if (lane == 0) red[warp * NP + p] = v;
    }
    __syncthreads();
    if (warp == 0) {
#pragma unroll
        for (int p = 0; p < NP; p++) {
            X v = lane < nwarps ? red[lane * NP + p] : FP::x_zero();
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) v = FP::x_add(v, FP::x_shfl_down(v, off));
            if (lane == 0) out[p] = v;
        }
    }
    __syncthreads();
}

// One layer is split over `groups` CTAs by terms (h is linear in them): CTA g keeps its own copy of t_0 (slot 0) and the tables of
// its terms (slots 1 + 2k, 2 + 2k = l, r of term i0 + k) in shared memory, writes its partial sums per round to gpart, and the last
// CTA of the layer to finish (counter) adds the groups up into the message slots. One CTA per layer took 60 us for 35 layers
// (profiles/r2_launch_list.md): a serial chain of rounds with 2 (term, pair) items per thread in its first round.
template <class FP> __global__ void __launch_bounds__(HG_TAIL_THREADS) k_gp_tail(const GpTailItem<FP>* __restrict__ items, int max_groups) {
    typedef typename FP::B B;
    typedef typename FP::X X;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ bool is_last;
    const GpTailItem<FP> it = items[blockIdx.x / max_groups];
    const int g = blockIdx.x % max_groups;
    if (g >= it.groups) return;
    const int i0 = it.i_begin + g * it.tpg, i1 = min(it.i_end, i0 + it.tpg);
    const int nt = i1 - i0, ntab = 1 + 2 * nt, cap = 1 + 2 * it.tpg;
    int len = it.n;
    X* A = reinterpret_cast<X*>(smem_raw);        // [cap][n]
    X* Bf = A + (size_t)cap * len;                 // [cap][n / 2]
    X* red = Bf + (size_t)cap * (len / 2);         // [32][4]
    X* gpart = it.gpart + (size_t)g * (HG_GP_TAIL_MAXR + 1) * 4;  // slot 0 = round 0 (from_base), slot 1 + k = k-th sampled tail round
    if (it.from_base) {
        const B* base = (const B*)it.in;  // vector i = [l_i (n) | r_i (n)] -> tables 2i, 2i+1 are consecutive runs of n
        for (int e = threadIdx.x; e < ntab * len; e += blockDim.x) {
            const int slot = e / len, k = e % len;
            const size_t tab = slot ? (size_t)(2 * i0 + slot - 1) : 0;
            A[e] = FP::lift(base[tab * len + k]);
        }
        __syncthreads();
        // round 0 on the unscaled tables: h(0), h(inf), h(-1), h(1)
        X acc[4] = {FP::x_zero(), FP::x_zero(), FP::x_zero(), FP::x_zero()};
        const int npairs = len / 2;
        for (int e = threadIdx.x; e < nt * npairs; e += blockDim.x) {
            const int k = e / npairs, b = e % npairs;
            const X t_lo = A[2 * b], t_hi = A[2 * b + 1];
            const X l_lo = A[(1 + 2 * k) * len + 2 * b], l_hi = A[(1 + 2 * k) * len + 2 * b + 1];
            const X r_lo = A[(2 + 2 * k) * len + 2 * b], r_hi = A[(2 + 2 * k) * len + 2 * b + 1];
            const X ci = it.c[i0 + k];
            acc[0] = FP::x_add(acc[0], FP::fmul(FP::fmul(ci, t_lo), FP::fmul(l_lo, r_lo)));
            acc[1] = FP::x_add(acc[1], FP::fmul(FP::fmul(ci, FP::slope(t_lo, t_hi)), FP::fmul(FP::slope(l_lo, l_hi), FP::slope(r_lo, r_hi))));
            acc[2] = FP::x_add(acc[2], FP::fmul(FP::fmul(ci, FP::at_m1(t_lo, t_hi)), FP::fmul(FP::at_m1(l_lo, l_hi), FP::at_m1(r_lo, r_hi))));
            acc[3] = FP::x_add(acc[3], FP::fmul(FP::fmul(ci, t_hi), FP::fmul(l_hi, r_hi)));
        }
        tail_block_sum<FP, 4>(acc, red, gpart);
        // pre-scale l_i by c_i (i > 0) and r_0 by c_0, as round 1 of the streaming kernels does (slot 0, the copy of t_0, stays)
        for (int e = threadIdx.x; e < nt * len; e += blockDim.x) {
            const int k = e / len, q = e % len, i = i0 + k, slot = i ? 1 + 2 * k : 2 + 2 * k;
            A[slot * len + q] = FP::fmul(A[slot * len + q], it.c[i]);
        }
        __syncthreads();
    } else {
        const X* src = (const X*)it.in;
        for (int e = threadIdx.x; e < ntab * len; e += blockDim.x) {
            const int slot = e / len, k = e % len;
            const size_t tab = slot ? (size_t)(2 * i0 + slot - 1) : 0;
            A[e] = src[tab * len + k];
        }
        if (g == 0 && it.r0n > 0) {  // round 0 was sampled while the tree was built: add up the CTA partials
            X acc[4] = {FP::x_zero(), FP::x_zero(), FP::x_zero(), FP::x_zero()};
            for (int b = threadIdx.x; b < it.r0n; b += blockDim.x)
#pragma unroll
                for (int p = 0; p < 4; p++) acc[p] = FP::x_add(acc[p], it.r0part[(size_t)b * 4 + p]);
            tail_block_sum<FP, 4>(acc, red, it.msg0);
        }
        __syncthreads();
    }
    X* cur = A;
    X* nxt = Bf;
    const int pre = it.from_base ? 0 : 1;
    if (pre) {  // the last streamed round wrote its tables folded by its own challenge: sample the first tail round on them as they are
        const int npairs = len / 2;
        X acc[3] = {FP::x_zero(), FP::x_zero(), FP::x_zero()};
        for (int e = threadIdx.x; e < nt * npairs; e += blockDim.x) {
            const int k = e / npairs, b = e % npairs;
            const X* t = cur + 2 * b;
            const X* l = cur + (1 + 2 * k) * len + 2 * b;
            const X* q = cur + (2 + 2 * k) * len + 2 * b;
            const X p0 = FP::fmul(l[0], q[0]), p1 = FP::fmul(FP::slope(l[0], l[1]), FP::slope(q[0], q[1])),
                    p2 = FP::fmul(FP::at_m1(l[0], l[1]), FP::at_m1(q[0], q[1]));
            acc[0] = FP::x_add(acc[0], FP::fmul(t[0], p0));
            acc[1] = FP::x_add(acc[1], FP::fmul(FP::slope(t[0], t[1]), p1));
            acc[2] = FP::x_add(acc[2], FP::fmul(FP::at_m1(t[0], t[1]), p2));
        }
        tail_block_sum<FP, 3>(acc, red, gpart + 4);
    }
    for (int rd = 0; rd < it.rounds; rd++) {
        const X r = it.chal[rd];
        const typename FP::FoldAux aux = FP::fold_aux(r);
        const int npairs = len / 4, half = len / 2;
        X acc[3] = {FP::x_zero(), FP::x_zero(), FP::x_zero()};
        for (int b = threadIdx.x; b < npairs; b += blockDim.x) {  // this CTA's copy of t_0
            const X* t = cur + 4 * b;
            nxt[2 * b] = FP::fold(t[0], t[1], r, aux);
            nxt[2 * b + 1] = FP::fold(t[2], t[3], r, aux);
        }
        for (int e = threadIdx.x; e < nt * npairs; e += blockDim.x) {
            const int k = e / npairs, b = e % npairs;
            const X* t = cur + 4 * b;
            const X* l = cur + (1 + 2 * k) * len + 4 * b;
            const X* q = cur + (2 + 2 * k) * len + 4 * b;
            const X t_lo = FP::fold(t[0], t[1], r, aux), t_hi = FP::fold(t[2], t[3], r, aux);
            const X l_lo = FP::fold(l[0], l[1], r, aux), l_hi = FP::fold(l[2], l[3], r, aux);
            const X r_lo = FP::fold(q[0], q[1], r, aux), r_hi = FP::fold(q[2], q[3], r, aux);
            nxt[(1 + 2 * k) * half + 2 * b] = l_lo;
            nxt[(1 + 2 * k) * half + 2 * b + 1] = l_hi;
            nxt[(2 + 2 * k) * half + 2 * b] = r_lo;
            nxt[(2 + 2 * k) * half + 2 * b + 1] = r_hi;
            const X p0 = FP::fmul(l_lo, r_lo), p1 = FP::fmul(FP::slope(l_lo, l_hi), FP::slope(r_lo, r_hi)),
                    p2 = FP::fmul(FP::at_m1(l_lo, l_hi), FP::at_m1(r_lo, r_hi));
            acc[0] = FP::x_add(acc[0], FP::fmul(t_lo, p0));
            acc[1] = FP::x_add(acc[1], FP::fmul(FP::slope(t_lo, t_hi), p1));
            acc[2] = FP::x_add(acc[2], FP::fmul(FP::at_m1(t_lo, t_hi), p2));
        }
        tail_block_sum<FP, 3>(acc, red, gpart + (size_t)(1 + pre + rd) * 4);  // ends with __syncthreads: nxt is complete
        X* tmp = cur; cur = nxt; nxt = tmp;
        len = half;
    }
    // len == 2: final evaluations of this CTA's tables
    {
        const X r = it.chal[it.rounds];
        const typename FP::FoldAux aux = FP::fold_aux(r);
        for (int s = 1 + threadIdx.x; s < ntab; s += blockDim.x) it.evals[2 * i0 + s - 1] = FP::fold(cur[2 * s], cur[2 * s + 1], r, aux);
    }
    // the last CTA of the layer adds the groups up
    if (threadIdx.x == 0) {
        __threadfence();
        const unsigned t = atomicAdd(it.counter, 1u);
        is_last = (t == (unsigned)it.groups - 1);
    }
    __syncthreads();
    if (!is_last) return;
    __threadfence();
    for (int e = threadIdx.x; e < (1 + pre + it.rounds) * 4; e += blockDim.x) {
        const int slot = e / 4, p = e % 4;
        if (slot == 0 ? !it.from_base : p == 3) continue;
        X v = FP::x_zero();
        for (int q = 0; q < it.groups; q++) v = FP::x_add(v, FP::x_ldcg(it.gpart + ((size_t)q * (HG_GP_TAIL_MAXR + 1) + slot) * 4 + p));
        if (slot == 0) it.msg0[p] = v; else it.msg[3 * (slot - 1) + p] = v;
    }
    if (threadIdx.x == 0) *it.counter = 0;
}

}  // namespace hg
