// K11/K12: kernels for the generic GKR layers (Vanilla / FFT nodes of /root/reference/bfv-gkr/src/sk_encryption_circuit.rs:86-293;
// the engine itself is the un-vendored `gkr` crate, restated in DESIGN.md section 3). Every layer reduces to a product sumcheck
//        sum_x W[x] * prod_{k<nt} T_k[x]            nt = 1 (linear / FFT layers), nt = 2 (element-wise product layer)
// where W is an extension-field weight table derived from the claim points (eq tables pushed through the wiring or the FFT
// matrix) and T_k are the node's input tables. With prefetched challenges all nodes are independent, so round j of every
// node runs in ONE launch (descriptor table, like gp_kernels.cuh).
#pragma once
#include "gp_kernels.cuh"

namespace hg {

// ---- forward evaluation of a Vanilla layer: out[r*ng + g] = c_g + sum coef * in_k[r*sub + w] + sum coef * in*in
struct VanillaFwd {
    const u64* add_ptr;   // [ng + 1]
    const u32* add_in;    // input index
    const u64* add_wire;
    const u64* mul_ptr;   // [ng + 1]
    const u32* mul_in0; const u64* mul_w0; const u32* mul_in1; const u64* mul_w1;
};
template <class FP>
__global__ void k_vanilla_eval(VanillaFwd w, const typename FP::B* __restrict__ add_coef, const typename FP::B* __restrict__ mul_coef,
                               const typename FP::B* __restrict__ consts, const typename FP::B* const* __restrict__ inputs, size_t ng,
                               size_t sub, int num_reps, size_t out_len, typename FP::B* __restrict__ out) {
    typedef typename FP::B B;
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= out_len) return;
    if (t >= ng * num_reps) { out[t] = FP::b_zero(); return; }
    const size_t r = t / ng, g = t % ng;
    // unreduced sum of products, one reduction per gate
    typename FP::BAcc acc = FP::bacc_zero();
    for (u64 e = w.add_ptr[g]; e < w.add_ptr[g + 1]; e++) FP::bacc_mad(acc, add_coef[e], inputs[w.add_in[e]][r * sub + w.add_wire[e]]);
    for (u64 e = w.mul_ptr[g]; e < w.mul_ptr[g + 1]; e++)
        FP::bacc_mad(acc, mul_coef[e], FP::fmul(inputs[w.mul_in0[e]][r * sub + w.mul_w0[e]], inputs[w.mul_in1[e]][r * sub + w.mul_w1[e]]));
    out[t] = FP::b_add(consts[g], FP::bacc_reduce(acc));
}

// Forward evaluation of the layers whose gates come in runs: gates g0..g0+n-1 each read wire w0_e + (g - g0) of input in_e with one
// coefficient per edge slot e (relay / scale / shift / sum layers: one to five slots, sk_encryption_circuit.rs:97-285), or multiply two
// inputs element-wise (ne = -2, :245-260). One streamed launch per circuit level for all such layers instead of one index-chasing
// launch per layer (k_vanilla_eval: 28 bytes of gate description per edge). Same products, one reduction per gate: identical values.
constexpr int HG_FWD_MAXE = 5;
constexpr int HG_FWD_PER_THREAD = 4;
template <class FP> struct FwdRunItem {
    typename FP::B* out;
    u64 n;
    const typename FP::B* in[HG_FWD_MAXE];
    typename FP::B coef[HG_FWD_MAXE];
    typename FP::B cst;
    int ne;  // additive edge slots (0: constant gates), -2: out = in[0] * in[1]
    int blk_start;
};
template <class FP> __global__ void k_vanilla_runs(const FwdRunItem<FP>* __restrict__ items, int nitems) {
    typedef typename FP::B B;
    const FwdRunItem<FP> it = items[find_item(items, nitems)];
    const size_t base = (size_t)(blockIdx.x - it.blk_start) * blockDim.x * HG_FWD_PER_THREAD + threadIdx.x;
#pragma unroll
    for (int k = 0; k < HG_FWD_PER_THREAD; k++) {
        const size_t i = base + (size_t)k * blockDim.x;
        if (i >= it.n) continue;
        typename FP::BAcc acc = FP::bacc_zero();
        if (it.ne == -2) FP::bacc_mad(acc, FP::b_one(), FP::fmul(it.in[0][i], it.in[1][i]));
        else for (int e = 0; e < it.ne; e++) FP::bacc_mad(acc, it.coef[e], it.in[e][i]);
        it.out[i] = FP::b_add(it.cst, FP::bacc_reduce(acc));
    }
}

// ---- eq factor tables of every (node, claim) pair in one launch
// eq_lo of claim t carries the factor alpha^t (alpha = nullptr: single claim), so W = sum_t eq_lo_t (x) eq_hi_t needs no scaling pass
template <class FP> struct EqSplitItem {
    const typename FP::X* point; typename FP::X* eq_lo; typename FP::X* eq_hi; const typename FP::X* alpha;
    int nv, lo_bits, blk_start, t;
};
template <class FP> __global__ void k_eq_split_multi(const EqSplitItem<FP>* __restrict__ items, int nitems) {
    typedef typename FP::X X;
    const EqSplitItem<FP> it = items[find_item(items, nitems)];
    const size_t t = (size_t)(blockIdx.x - it.blk_start) * blockDim.x + threadIdx.x;
    const size_t nlo = (size_t)1 << it.lo_bits, nhi = (size_t)1 << (it.nv - it.lo_bits);
    if (t >= nlo + nhi) return;
    const bool hi = t >= nlo;
    const size_t k = hi ? t - nlo : t;
    const int first = hi ? it.lo_bits : 0, last = hi ? it.nv : it.lo_bits;
    X acc = FP::x_one();
    if (!hi && it.alpha) { const X a = *it.alpha; for (int q = 0; q < it.t; q++) acc = FP::fmul(acc, a); }
    for (int i = first; i < last; i++) {
        X r = it.point[i];
        X f = ((k >> (i - first)) & 1) ? r : FP::x_sub(FP::x_one(), r);
        acc = FP::fmul(acc, f);
    }
    (hi ? it.eq_hi : it.eq_lo)[k] = acc;
}

// ---- W = sum_t alpha^t * eq(z_t, .) for every node in one launch; the factor tables of a node's claims lie back to back
// ([eq_lo_t | eq_hi_t], stride elements apart), alpha^t is already in eq_lo_t
template <class FP> struct EqAccItem {
    const typename FP::X* eq0;   // eq_lo of claim 0
    typename FP::X* w;
    u64 n, stride;
    int lo_bits, n_claims, blk_start;
};
constexpr int HG_EQACC_PER_THREAD = 8;  // one element per thread made the launch block-dispatch bound (47 616 CTAs, 230 us)
template <class FP> __global__ void k_eq_accumulate(const EqAccItem<FP>* __restrict__ items, int nitems) {
    typedef typename FP::X X;
    const EqAccItem<FP> it = items[find_item(items, nitems)];
    const size_t nlo = (size_t)1 << it.lo_bits;
    const size_t base = (size_t)(blockIdx.x - it.blk_start) * blockDim.x * HG_EQACC_PER_THREAD + threadIdx.x;
    if (it.n_claims == 1) {  // almost every node: all loads first, then the products
        X lo[HG_EQACC_PER_THREAD], hi[HG_EQACC_PER_THREAD];
#pragma unroll
        for (int k = 0; k < HG_EQACC_PER_THREAD; k++) {
            const size_t i = base + (size_t)k * blockDim.x;
            lo[k] = hi[k] = FP::x_zero();
            if (i < it.n) { lo[k] = it.eq0[i & (nlo - 1)]; hi[k] = it.eq0[nlo + (i >> it.lo_bits)]; }
        }
#pragma unroll
        for (int k = 0; k < HG_EQACC_PER_THREAD; k++) {
            const size_t i = base + (size_t)k * blockDim.x;
            if (i < it.n) it.w[i] = FP::fmul(lo[k], hi[k]);
        }
        return;
    }
#pragma unroll 2
    for (int k = 0; k < HG_EQACC_PER_THREAD; k++) {
        const size_t i = base + (size_t)k * blockDim.x;
        if (i >= it.n) return;
        const size_t lo = i & (nlo - 1), hi = i >> it.lo_bits;
        typename FP::XAcc a = FP::xacc_zero_();
        for (int t = 0; t < it.n_claims; t++) {
            const X* e = it.eq0 + (size_t)t * it.stride;
            FP::xacc_mad_(a, e[lo], e[nlo + hi]);
        }
        it.w[i] = FP::xacc_reduce_(a);
    }
}

// ---- A[x] = sum_{(o, c) in rev[x]} c * W[o]  (weights pushed through the wiring, reverse CSR), const = sum_g W[g] c_g
template <class FP> struct WiringItem {
    const u64* rev_ptr; const u32* rev_out; const typename FP::B* rev_coef; const typename FP::X* w; typename FP::X* A;
    u64 n; int blk_start;
};
constexpr int HG_WIRING_PER_THREAD = 4;  // independent pointer-chasing chains per thread (ptr -> edge -> W): memory-level parallelism
template <class FP> __global__ void k_wiring_gather(const WiringItem<FP>* __restrict__ items, int nitems) {
    const WiringItem<FP> it = items[find_item(items, nitems)];
    const size_t base = (size_t)(blockIdx.x - it.blk_start) * blockDim.x * HG_WIRING_PER_THREAD + threadIdx.x;
    u64 e0[HG_WIRING_PER_THREAD], e1[HG_WIRING_PER_THREAD];
#pragma unroll
    for (int k = 0; k < HG_WIRING_PER_THREAD; k++) {
        const size_t x = base + (size_t)k * blockDim.x;
        e0[k] = e1[k] = 0;
        if (x < it.n) { e0[k] = it.rev_ptr[x]; e1[k] = it.rev_ptr[x + 1]; }
    }
#pragma unroll
    for (int k = 0; k < HG_WIRING_PER_THREAD; k++) {
        const size_t x = base + (size_t)k * blockDim.x;
        if (x >= it.n) continue;
        typename FP::XAcc acc = FP::xacc_zero_();
        for (u64 e = e0[k]; e < e1[k]; e++) FP::xacc_mad_b(acc, it.w[it.rev_out[e]], it.rev_coef[e]);
        it.A[x] = FP::xacc_reduce_(acc);
    }
}
// Linear layers whose reverse wiring is piecewise the identity: every input element feeds at most one output and consecutive elements
// feed consecutive outputs with the same coefficient (the relay / scale / shift / sum layers of sk_encryption_circuit.rs:97-285). Then
// A = coef * W run by run, streamed, instead of chasing rev_ptr -> rev_out -> W per element (k_wiring_gather: 228 us, 0.44 GB of
// index reads per proof, profiles/r2_launch_list.md). Same products, same reduction: identical field elements.
template <class FP> struct WireRunItem {
    const typename FP::X* w;  // W + first output of the run
    typename FP::X* A;        // A + first input element of the run
    u64 n;
    typename FP::B coef;
    int kind;                 // 0: elements that feed nothing (zeros), 1: coefficient one (copy), 2: scaled
    int blk_start;
};
constexpr int HG_WIRERUN_PER_THREAD = 4;
template <class FP> __global__ void k_wiring_runs(const WireRunItem<FP>* __restrict__ items, int nitems) {
    typedef typename FP::X X;
    const WireRunItem<FP> it = items[find_item(items, nitems)];
    const size_t base = (size_t)(blockIdx.x - it.blk_start) * blockDim.x * HG_WIRERUN_PER_THREAD + threadIdx.x;
    X v[HG_WIRERUN_PER_THREAD];
#pragma unroll
    for (int k = 0; k < HG_WIRERUN_PER_THREAD; k++) {
        const size_t i = base + (size_t)k * blockDim.x;
        v[k] = FP::x_zero();
        if (it.kind != 0 && i < it.n) v[k] = it.w[i];
    }
#pragma unroll
    for (int k = 0; k < HG_WIRERUN_PER_THREAD; k++) {
        const size_t i = base + (size_t)k * blockDim.x;
        if (i >= it.n) continue;
        if (it.kind == 2) {
            typename FP::XAcc acc = FP::xacc_zero_();
            FP::xacc_mad_b(acc, v[k], it.coef);
            v[k] = FP::xacc_reduce_(acc);
        }
        it.A[i] = v[k];
    }
}
// ---- general layers (the two-phase layer sumcheck, DESIGN.md section 3, A11). The product terms are two reverse CSRs over the
// S entries of the concatenated inputs X (num_reps expanded): row x of the x-keyed CSR holds (y, output, coefficient) of every term
// W-weighted as W[output] coef X[x] X[y], row y of the y-keyed CSR the same terms with their x. Gathers: no atomics.
template <class FP> struct GeneralItem {
    const u64* ptr; const u32* other; const u32* out; const typename FP::B* coef;
    const typename FP::X* w;                                       // W: weights of the outputs
    const typename FP::B* tab;                                     // X (phase 1)
    const typename FP::X* eq_lo; const typename FP::X* eq_hi;      // eq(u, .) = eq_lo[x mod 2^lo_bits] eq_hi[x >> lo_bits] (phase 2)
    typename FP::X* dst;                                           // phase 1: A, turned into G = A + H in place; phase 2: M_u
    u64 n; int lo_bits, blk_start;
};
constexpr int HG_GENERAL_PER_THREAD = 4;  // independent row chains per thread (ptr -> term -> W): memory-level parallelism
// phase 1: G[x] = A[x] + H[x],  H[x] = sum_{(y, o, c) in row x} W[o] c X[y]
template <class FP> __global__ void k_general_g(const GeneralItem<FP>* __restrict__ items, int nitems) {
    const GeneralItem<FP> it = items[find_item(items, nitems)];
    const size_t base = (size_t)(blockIdx.x - it.blk_start) * blockDim.x * HG_GENERAL_PER_THREAD + threadIdx.x;
    u64 e0[HG_GENERAL_PER_THREAD], e1[HG_GENERAL_PER_THREAD];
#pragma unroll
    for (int k = 0; k < HG_GENERAL_PER_THREAD; k++) {
        const size_t x = base + (size_t)k * blockDim.x;
        e0[k] = e1[k] = 0;
        if (x < it.n) { e0[k] = it.ptr[x]; e1[k] = it.ptr[x + 1]; }
    }
#pragma unroll
    for (int k = 0; k < HG_GENERAL_PER_THREAD; k++) {
        const size_t x = base + (size_t)k * blockDim.x;
        if (x >= it.n || e0[k] == e1[k]) continue;
        typename FP::XAcc acc = FP::xacc_zero_();
        for (u64 e = e0[k]; e < e1[k]; e++) FP::xacc_mad_b(acc, it.w[it.out[e]], FP::fmul(it.coef[e], it.tab[it.other[e]]));
        it.dst[x] = FP::x_add(it.dst[x], FP::xacc_reduce_(acc));
    }
}
// phase 2: M_u[y] = sum_{(x, o, c) in row y} eq(u, x) W[o] c
template <class FP> __global__ void k_general_mu(const GeneralItem<FP>* __restrict__ items, int nitems) {
    typedef typename FP::X X;
    const GeneralItem<FP> it = items[find_item(items, nitems)];
    const size_t base = (size_t)(blockIdx.x - it.blk_start) * blockDim.x * HG_GENERAL_PER_THREAD + threadIdx.x;
    const size_t mask = ((size_t)1 << it.lo_bits) - 1;
    u64 e0[HG_GENERAL_PER_THREAD], e1[HG_GENERAL_PER_THREAD];
#pragma unroll
    for (int k = 0; k < HG_GENERAL_PER_THREAD; k++) {
        const size_t y = base + (size_t)k * blockDim.x;
        e0[k] = e1[k] = 0;
        if (y < it.n) { e0[k] = it.ptr[y]; e1[k] = it.ptr[y + 1]; }
    }
#pragma unroll
    for (int k = 0; k < HG_GENERAL_PER_THREAD; k++) {
        const size_t y = base + (size_t)k * blockDim.x;
        if (y >= it.n) continue;
        typename FP::XAcc acc = FP::xacc_zero_();
        for (u64 e = e0[k]; e < e1[k]; e++) {
            const size_t x = it.other[e];
            const X eqx = FP::fmul(it.eq_lo[x & mask], it.eq_hi[x >> it.lo_bits]);
            FP::xacc_mad_b(acc, FP::fmul(eqx, it.w[it.out[e]]), it.coef[e]);
        }
        it.dst[y] = FP::xacc_reduce_(acc);
    }
}
// concatenated input tables of the layer sumchecks: dst[0..n) = src[0..n) (src = nullptr: zeros), every node's pieces in one launch
template <class FP> struct ConcatItem { const typename FP::B* src; typename FP::B* dst; u64 n; int blk_start; };
constexpr int HG_CONCAT_PER_THREAD = 8;
template <class FP> __global__ void k_concat_items(const ConcatItem<FP>* __restrict__ items, int nitems) {
    const ConcatItem<FP> it = items[find_item(items, nitems)];
    const size_t base = (size_t)(blockIdx.x - it.blk_start) * blockDim.x * HG_CONCAT_PER_THREAD + threadIdx.x;
#pragma unroll
    for (int k = 0; k < HG_CONCAT_PER_THREAD; k++) {
        const size_t i = base + (size_t)k * blockDim.x;
        if (i < it.n) it.dst[i] = it.src ? it.src[i] : FP::b_zero();
    }
}

// tabs[q] = extension table of node q (n elements); planes = [PLANES*q + p][n]
template <class FP> __global__ void k_ext_split(typename FP::X* const* __restrict__ tabs, size_t n, typename FP::B* __restrict__ planes) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const size_t q = blockIdx.y;
    typename FP::X v = tabs[q][i];
#pragma unroll
    for (int p = 0; p < FP::PLANES; p++) planes[(FP::PLANES * q + p) * n + i] = FP::plane(v, p);
}
template <class FP> __global__ void k_ext_merge(const typename FP::B* __restrict__ planes, size_t n, typename FP::X* const* __restrict__ tabs) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const size_t q = blockIdx.y;
    typename FP::B b[FP::PLANES];
#pragma unroll
    for (int p = 0; p < FP::PLANES; p++) b[p] = planes[(FP::PLANES * q + p) * n + i];
    tabs[q][i] = FP::from_planes(b);
}

// ---- product sumcheck rounds, all nodes per launch. msg slots per round: [h(0), h(inf), h(-1), h(1)] (h(-1) only for nt = 2,
// h(1) only in round 0; unused slots are written as zero)
template <class FP> struct ProdItem {
    const typename FP::X* w_in; typename FP::X* w_out;
    const void* tab_in; typename FP::X* tab_out;   // nt tables of n_in elements back to back
    u64 n_in;
    const typename FP::X* r_prev;
    typename FP::X* msg; typename FP::X* partials; unsigned* counter;
    int nt, blk_start, nblk, bx;
};
// one item, NT tables. Threads run few iterations here, so sums are kept reduced (4 registers each): unreduced accumulators
// (24 registers each) cost more in occupancy than they save in reductions (measured: 2.5 ms vs 1.8 ms per proof)
// FUSE0 (round 1 in prefetch mode, TIN = base): r_0 is known before round 0 is computed, so the pass that folds the raw tables by
// r_0 also samples round 0 on them (a quad of raw entries = two round-0 pairs) and the launch of round 0, one more read of the
// largest tables of the class, is gone. acc[0..3] = round 0 [h(0), h(inf), h(-1), h(1)], acc[4..7] = round 1.
template <class FP, class TIN, bool FOLD, int NT, bool FUSE0 = false>
__device__ __forceinline__ void prod_round_item(const ProdItem<FP>& it, unsigned lb, typename FP::X (&acc)[FUSE0 ? 8 : 4]) {
    typedef typename FP::X X;
    typedef typename std::conditional<FOLD, X, TIN>::type EL;
    constexpr int NS = NT + 1;  // samples 0, inf (and -1 for the degree-3 case); slot 3 = h(1), round 0 only
    const TIN* tab = (const TIN*)it.tab_in;
    const size_t n_in = it.n_in, npairs = FOLD ? n_in / 4 : n_in / 2, n_out = n_in / 2;
    X r = FP::x_zero();
    typename FP::FoldAux aux;
    if (FOLD) { r = *it.r_prev; aux = FP::fold_aux(r); }
    (void)NS;
    if constexpr (NT == 1 && !FOLD) {
        // round 0 of a degree-2 node (most of the bytes of the class): extension weight times BASE table entry, three samples,
        // unreduced accumulation (two 64x64 products per sample; 16 registers per accumulator because the X^2 column stays empty)
        typename FP::XAcc P0 = FP::xacc_zero_(), P1 = FP::xacc_zero_(), P3 = FP::xacc_zero_();
#pragma unroll 2
        for (size_t b = (size_t)lb * blockDim.x + threadIdx.x; b < npairs; b += (size_t)it.nblk * blockDim.x) {
            X w[2];
            TIN t[2];
            load2(it.w_in + 2 * b, w);
            load2(tab + 2 * b, t);
            FP::xacc_mad_b(P0, w[0], t[0]);
            FP::xacc_mad_b(P1, FP::slope(w[0], w[1]), FP::slope(t[0], t[1]));
            FP::xacc_mad_b(P3, w[1], t[1]);
        }
        acc[0] = FP::xacc_reduce_(P0); acc[1] = FP::xacc_reduce_(P1); acc[3] = FP::xacc_reduce_(P3);
        return;
    }
    constexpr int O = FUSE0 ? 4 : 0;  // where this round's samples go
    typename FP::XAcc Q0, Q1, Q3;     // FUSE0, NT == 1: round 0 = extension weight times BASE entry, accumulated unreduced as in the unfused round 0
    if constexpr (FUSE0 && NT == 1) { Q0 = FP::xacc_zero_(); Q1 = FP::xacc_zero_(); Q3 = FP::xacc_zero_(); }
    for (size_t b = (size_t)lb * blockDim.x + threadIdx.x; b < npairs; b += (size_t)it.nblk * blockDim.x) {
        X wlo, whi;
        X wraw[4];
        (void)wraw;
        if constexpr (FOLD) {
            X s[4];
            load4(it.w_in + 4 * b, s);
            if constexpr (FUSE0) { wraw[0] = s[0]; wraw[1] = s[1]; wraw[2] = s[2]; wraw[3] = s[3]; }
            wlo = FP::fold(s[0], s[1], r, aux); whi = FP::fold(s[2], s[3], r, aux);
            store2(it.w_out + 2 * b, wlo, whi);
        } else {
            X s[2];
            load2(it.w_in + 2 * b, s);
            wlo = s[0]; whi = s[1];
        }
        EL lo[NT], hi[NT];
        TIN traw[NT][4];
        (void)traw;
#pragma unroll
        for (int q = 0; q < NT; q++) {
            if constexpr (FOLD) {
                TIN s[4];
                load4(tab + (size_t)q * n_in + 4 * b, s);
                if constexpr (FUSE0) { traw[q][0] = s[0]; traw[q][1] = s[1]; traw[q][2] = s[2]; traw[q][3] = s[3]; }
                lo[q] = FP::fold(s[0], s[1], r, aux); hi[q] = FP::fold(s[2], s[3], r, aux);
                store2(it.tab_out + (size_t)q * n_out + 2 * b, lo[q], hi[q]);
            } else {
                TIN s[2];
                load2(tab + (size_t)q * n_in + 2 * b, s);
                lo[q] = s[0]; hi[q] = s[1];
            }
        }
        if constexpr (FUSE0) {  // round 0 on the two raw pairs (0, 1) and (2, 3) of this quad
#pragma unroll
            for (int h = 0; h < 4; h += 2) {
                if constexpr (NT == 1) {
                    FP::xacc_mad_b(Q0, wraw[h], traw[0][h]);
                    FP::xacc_mad_b(Q1, FP::slope(wraw[h], wraw[h + 1]), FP::slope(traw[0][h], traw[0][h + 1]));
                    FP::xacc_mad_b(Q3, wraw[h + 1], traw[0][h + 1]);
                } else {
                    acc[0] = FP::x_add(acc[0], FP::fmul_any(wraw[h], FP::fmul(traw[0][h], traw[1][h])));
                    acc[1] = FP::x_add(acc[1], FP::fmul_any(FP::slope(wraw[h], wraw[h + 1]), FP::fmul(FP::slope(traw[0][h], traw[0][h + 1]), FP::slope(traw[1][h], traw[1][h + 1]))));
                    acc[2] = FP::x_add(acc[2], FP::fmul_any(FP::at_m1(wraw[h], wraw[h + 1]), FP::fmul(FP::at_m1(traw[0][h], traw[0][h + 1]), FP::at_m1(traw[1][h], traw[1][h + 1]))));
                    acc[3] = FP::x_add(acc[3], FP::fmul_any(wraw[h + 1], FP::fmul(traw[0][h + 1], traw[1][h + 1])));
                }
            }
        }
        if constexpr (NT == 1) {
            acc[O + 0] = FP::x_add(acc[O + 0], FP::fmul_any(wlo, lo[0]));
            acc[O + 1] = FP::x_add(acc[O + 1], FP::fmul_any(FP::slope(wlo, whi), FP::slope(lo[0], hi[0])));
            if (!FOLD) acc[3] = FP::x_add(acc[3], FP::fmul_any(whi, hi[0]));
        } else {
            acc[O + 0] = FP::x_add(acc[O + 0], FP::fmul_any(wlo, FP::fmul(lo[0], lo[1])));
            acc[O + 1] = FP::x_add(acc[O + 1], FP::fmul_any(FP::slope(wlo, whi), FP::fmul(FP::slope(lo[0], hi[0]), FP::slope(lo[1], hi[1]))));
            acc[O + 2] = FP::x_add(acc[O + 2], FP::fmul_any(FP::at_m1(wlo, whi), FP::fmul(FP::at_m1(lo[0], hi[0]), FP::at_m1(lo[1], hi[1]))));
            if (!FOLD) acc[3] = FP::x_add(acc[3], FP::fmul_any(whi, FP::fmul(hi[0], hi[1])));
        }
    }
    if constexpr (FUSE0 && NT == 1) { acc[0] = FP::xacc_reduce_(Q0); acc[1] = FP::xacc_reduce_(Q1); acc[3] = FP::xacc_reduce_(Q3); }
}
constexpr int HG_PROD_BLOCK = 128;  // threads per CTA of the streamed layer-sumcheck rounds
template <class FP, class TIN, bool FOLD, bool FUSE0 = false>
__global__ void __launch_bounds__(HG_PROD_BLOCK, ((FOLD || sizeof(typename FP::B) > 8) ? 1 : 3) * (HG_BLOCK / HG_PROD_BLOCK)) k_prod_round_multi(const ProdItem<FP>* __restrict__ items, int nitems) {
    typedef typename FP::X X;
    constexpr int NP = FUSE0 ? 8 : 4;  // FUSE0: it.msg is the slot of round 0, the slot of round 1 follows it
    const ProdItem<FP> it = items[find_item(items, nitems)];
    const unsigned lb = blockIdx.x - it.blk_start;
    X acc[NP];
#pragma unroll
    for (int p = 0; p < NP; p++) acc[p] = FP::x_zero();
    if (it.nt == 1) prod_round_item<FP, TIN, FOLD, 1, FUSE0>(it, lb, acc);
    else prod_round_item<FP, TIN, FOLD, 2, FUSE0>(it, lb, acc);
    block_reduce_finalize_ex<FP, NP>(acc, it.partials, it.counter, it.msg, it.nblk, lb);
}

// ---- the last rounds of every node sumcheck in ONE launch: one CTA per node, weights and tables (extension elements, at most
// 2^(HG_PROD_TAIL_LOG+1) entries each) in shared memory. Replaces ~10 launches of a few microseconds of work each.
constexpr int HG_PROD_TAIL_LOG = 9;
template <class FP> struct ProdTailItem {
    const typename FP::X* w_in; const typename FP::X* tab_in;   // output of streaming round rt-1: n_in entries each (nt tables back to back)
    const typename FP::X* chal;                                  // r_{rt-1} .. r_{nv-1}
    typename FP::X* msg;                                         // slot of round rt (4 per round)
    typename FP::X* evals;
    const typename FP::X* capture;                               // linear layers whose capture round ran in the streaming part, else nullptr
    int n_in, nt, rounds, linear, arity, cap_round;              // cap_round: index (0-based within the tail) of the round whose folded table holds the input evaluations, -1: none
    const typename FP::X* mid_part;                              // rounds done by k_prod_mid_one before this tail: CTA partial sums [mid_rounds][mid_nseg][4] ...
    typename FP::X* mid_msg;                                     // ... summed into the 4 message slots of each of those rounds (nullptr: no mid stage)
    int mid_nseg, mid_rounds;
};
template <class FP> __device__ __forceinline__ void prod_tail_body(const ProdTailItem<FP>& it, unsigned char* smem_raw) {
    typedef typename FP::X X;
    const int nt = it.nt, ntab = nt + 1;
    int len = it.n_in;
    X* cur = reinterpret_cast<X*>(smem_raw);            // [ntab][n_in]: table 0 = weights
    X* nxt = cur + (size_t)ntab * it.n_in;              // [ntab][n_in/2]
    X* red = nxt + (size_t)ntab * (it.n_in / 2);        // [32][3]
    for (int e = threadIdx.x; e < len; e += blockDim.x) cur[e] = it.w_in[e];
    for (int e = threadIdx.x; e < nt * len; e += blockDim.x) cur[len + e] = it.tab_in[e];
    if (it.mid_msg)  // the messages of the rounds k_prod_mid_one ran: add up its CTA partials (field addition is exact: any order)
        for (int t = threadIdx.x; t < 4 * it.mid_rounds; t += blockDim.x) {
            const int rd = t >> 2, p = t & 3;
            X s = FP::x_zero();
            if (p < 3) for (int g = 0; g < it.mid_nseg; g++) s = FP::x_add(s, it.mid_part[((size_t)rd * it.mid_nseg + g) * 4 + p]);
            it.mid_msg[t] = s;
        }
    __syncthreads();
    for (int rd = 0; rd < it.rounds; rd++) {
        const X r = it.chal[rd];
        const typename FP::FoldAux aux = FP::fold_aux(r);
        const int npairs = len / 4, half = len / 2;
        X acc[3] = {FP::x_zero(), FP::x_zero(), FP::x_zero()};
        for (int b = threadIdx.x; b < npairs; b += blockDim.x) {
            X lo[3], hi[3];
            for (int q = 0; q < ntab; q++) {
                const X* s = cur + (size_t)q * len + 4 * b;
                lo[q] = FP::fold(s[0], s[1], r, aux); hi[q] = FP::fold(s[2], s[3], r, aux);
                nxt[(size_t)q * half + 2 * b] = lo[q]; nxt[(size_t)q * half + 2 * b + 1] = hi[q];
            }
            if (nt == 1) {
                acc[0] = FP::x_add(acc[0], FP::fmul(lo[0], lo[1]));
                acc[1] = FP::x_add(acc[1], FP::fmul(FP::slope(lo[0], hi[0]), FP::slope(lo[1], hi[1])));
            } else {
                acc[0] = FP::x_add(acc[0], FP::fmul(lo[0], FP::fmul(lo[1], lo[2])));
                acc[1] = FP::x_add(acc[1], FP::fmul(FP::slope(lo[0], hi[0]), FP::fmul(FP::slope(lo[1], hi[1]), FP::slope(lo[2], hi[2]))));
                acc[2] = FP::x_add(acc[2], FP::fmul(FP::at_m1(lo[0], hi[0]), FP::fmul(FP::at_m1(lo[1], hi[1]), FP::at_m1(lo[2], hi[2]))));
            }
        }
        tail_block_sum<FP, 3>(acc, red, it.msg + 4 * (size_t)rd);  // ends with a barrier: nxt is complete
        if (threadIdx.x == 0) it.msg[4 * (size_t)rd + 3] = FP::x_zero();
        if (rd == it.cap_round)  // linear layer: the table folded over the low variables holds the evaluations of the inputs
            for (int kk = threadIdx.x; kk < it.arity; kk += blockDim.x) it.evals[kk] = nxt[half + kk];
        X* t = cur; cur = nxt; nxt = t;
        len = half;
        __syncthreads();
    }
    // len == 2: final fold with the last challenge
    const X r = it.chal[it.rounds];
    const typename FP::FoldAux aux = FP::fold_aux(r);
    if (it.linear) {
        if (it.capture) { for (int kk = threadIdx.x; kk < it.arity; kk += blockDim.x) it.evals[kk] = it.capture[kk]; }
        else if (it.cap_round < 0 && threadIdx.x == 0) it.evals[0] = FP::fold(cur[len], cur[len + 1], r, aux);  // single input: its evaluation is the last fold
    } else {
        for (int q = threadIdx.x; q < nt; q += blockDim.x) it.evals[q] = FP::fold(cur[(size_t)(q + 1) * len], cur[(size_t)(q + 1) * len + 1], r, aux);
    }
}
// ---- the MIDDLE rounds of a product sumcheck in one launch: a CTA owns a segment of 2^(K+1) consecutive entries of every table
// (folding is local in the index: entries 2b, 2b+1 -> b), keeps it in shared memory, runs K rounds on it (fold by the previous
// challenge + sample, exactly the tail's loop) and leaves 2 entries per table and segment, plus its partial sums of the K round
// messages; the tail kernel of the job adds the partials up. Replaces K launches whose data fits the L2 anyway and whose time
// is launch latency (profiles/: ~11-18 us each) by one.
constexpr int HG_PROD_MID_K = 9;                        // rounds per launch; segment = 1024 entries
constexpr int HG_PROD_MID_SEG = 1 << (HG_PROD_MID_K + 1);
template <class FP> struct ProdMidItem {
    const typename FP::X* w_in; const typename FP::X* tab_in;   // n_in entries each (nt tables back to back), n_in = nseg * HG_PROD_MID_SEG
    typename FP::X* w_out; typename FP::X* tab_out;              // 2 * nseg entries each
    const typename FP::X* chal;                                  // chal[j]: challenge folded in round j of this stage
    typename FP::X* part;                                        // [K][nseg][4]
    typename FP::X* capture;                                     // linear layers whose capture round falls into this stage (else nullptr)
    unsigned long long n_in;
    int nt, nseg, cap_round, arity;
};
template <class FP> __device__ __forceinline__ void prod_mid_body(const ProdMidItem<FP>& it, const int seg, unsigned char* smem_raw) {
    typedef typename FP::X X;
    constexpr int K = HG_PROD_MID_K, S = HG_PROD_MID_SEG;
    const int nt = it.nt, ntab = nt + 1;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    X* cur = reinterpret_cast<X*>(smem_raw);            // [ntab][S]: table 0 = weights
    X* nxt = cur + (size_t)ntab * S;                    // [ntab][S/2]
    X* wred = nxt + (size_t)ntab * (S / 2);             // [K][nwarps][3]
    for (int e = threadIdx.x; e < S; e += blockDim.x) cur[e] = it.w_in[(size_t)seg * S + e];
    for (int q = 0; q < nt; q++)
        for (int e = threadIdx.x; e < S; e += blockDim.x) cur[(q + 1) * S + e] = it.tab_in[(size_t)q * it.n_in + (size_t)seg * S + e];
    __syncthreads();
    int len = S;
    for (int rd = 0; rd < K; rd++) {
        const X r = it.chal[rd];
        const typename FP::FoldAux aux = FP::fold_aux(r);
        const int npairs = len / 4, half = len / 2;
        X acc[3] = {FP::x_zero(), FP::x_zero(), FP::x_zero()};
        for (int b = threadIdx.x; b < npairs; b += blockDim.x) {
            X lo[3], hi[3];
            for (int q = 0; q < ntab; q++) {
                const X* s = cur + (size_t)q * len + 4 * b;
                lo[q] = FP::fold(s[0], s[1], r, aux); hi[q] = FP::fold(s[2], s[3], r, aux);
                nxt[(size_t)q * half + 2 * b] = lo[q]; nxt[(size_t)q * half + 2 * b + 1] = hi[q];
            }
            if (nt == 1) {
                acc[0] = FP::x_add(acc[0], FP::fmul(lo[0], lo[1]));
                acc[1] = FP::x_add(acc[1], FP::fmul(FP::slope(lo[0], hi[0]), FP::slope(lo[1], hi[1])));
            } else {
                acc[0] = FP::x_add(acc[0], FP::fmul(lo[0], FP::fmul(lo[1], lo[2])));
                acc[1] = FP::x_add(acc[1], FP::fmul(FP::slope(lo[0], hi[0]), FP::fmul(FP::slope(lo[1], hi[1]), FP::slope(lo[2], hi[2]))));
                acc[2] = FP::x_add(acc[2], FP::fmul(FP::at_m1(lo[0], hi[0]), FP::fmul(FP::at_m1(lo[1], hi[1]), FP::at_m1(lo[2], hi[2]))));
            }
        }
#pragma unroll
        for (int p = 0; p < 3; p++) {  // per-warp sums only: the cross-warp and cross-CTA sums happen once, at the end / in the tail
            X v = acc[p];
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) v = FP::x_add(v, FP::x_shfl_down(v, off));
            if (lane == 0) wred[((size_t)rd * nwarps + warp) * 3 + p] = v;
        }
        __syncthreads();  // nxt is complete
        if (rd == it.cap_round && it.capture)  // linear layer: the table folded over the low variables holds the evaluations of the inputs
            for (int kk = threadIdx.x; kk < half; kk += blockDim.x) { const size_t g = (size_t)seg * half + kk; if (g < (size_t)it.arity) it.capture[g] = nxt[half + kk]; }
        X* t = cur; cur = nxt; nxt = t;
        len = half;
    }
    // len == 2: the segment's pair of every table
    const size_t n_out = it.n_in >> K;
    for (int e = threadIdx.x; e < 2 * ntab; e += blockDim.x) {
        const int q = e >> 1, k = e & 1;
        X* dst = q == 0 ? it.w_out : it.tab_out + (size_t)(q - 1) * n_out;
        dst[2 * (size_t)seg + k] = cur[(size_t)q * 2 + k];
    }
    for (int t = threadIdx.x; t < 4 * K; t += blockDim.x) {
        const int rd = t >> 2, p = t & 3;
        X s = FP::x_zero();
        if (p < 3) for (int w = 0; w < nwarps; w++) s = FP::x_add(s, wred[((size_t)rd * nwarps + w) * 3 + p]);
        it.part[((size_t)rd * it.nseg + seg) * 4 + p] = s;
    }
}

// a single sumcheck (the Lasso collation sumcheck): descriptor by value
template <class FP> __global__ void __launch_bounds__(256) k_prod_mid_one(const ProdMidItem<FP> it) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    prod_mid_body<FP>(it, blockIdx.x, smem_raw);
}

template <class FP> __global__ void __launch_bounds__(256) k_prod_tail(const ProdTailItem<FP>* __restrict__ items) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    prod_tail_body<FP>(items[blockIdx.x], smem_raw);
}
// a single sumcheck (the Lasso collation sumcheck): descriptor by value
template <class FP> __global__ void __launch_bounds__(256) k_prod_tail_one(const ProdTailItem<FP> it) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    prod_tail_body<FP>(it, smem_raw);
}

// ---- streamed rounds of g = t_0 * t_1 on two tables laid out back to back (the Lasso collation sumcheck after the rewrite of
// DESIGN.md 2.1): fold with the previous challenge, write the folded pair of tables, sample h(0), h(inf) (and h(1) in round 0).
// Unreduced accumulation over HG_COLL_PER_THREAD pairs per thread. msg slots: [h(0), h(inf)] (+ [h(1)] in round 0).
constexpr int HG_COLL_PER_THREAD = 8;
template <class FP, class TIN, bool FOLD>
__global__ void __launch_bounds__(HG_BLOCK) k_coll_round(const TIN* __restrict__ in, typename FP::X* __restrict__ out, size_t n_in,
                                                       const typename FP::X* __restrict__ r_prev, typename FP::X* partials, unsigned* counter,
                                                       typename FP::X* msg) {
    typedef typename FP::X X;
    constexpr int NP = FOLD ? 2 : 3;
    const size_t npairs = FOLD ? n_in / 4 : n_in / 2, n_out = n_in / 2;
    X acc[NP];
    if constexpr (FOLD) {
        const X r = *r_prev;
        const typename FP::FoldAux aux = FP::fold_aux(r);
        typename FP::XAcc P0 = FP::xacc_zero_(), P1 = FP::xacc_zero_();
        for (size_t b = (size_t)blockIdx.x * blockDim.x + threadIdx.x; b < npairs; b += (size_t)gridDim.x * blockDim.x) {
            TIN q0[4], q1[4];
            load4(in + 4 * b, q0);
            load4(in + n_in + 4 * b, q1);
            const X lo0 = FP::fold(q0[0], q0[1], r, aux), hi0 = FP::fold(q0[2], q0[3], r, aux);
            const X lo1 = FP::fold(q1[0], q1[1], r, aux), hi1 = FP::fold(q1[2], q1[3], r, aux);
            store2(out + 2 * b, lo0, hi0);
            store2(out + n_out + 2 * b, lo1, hi1);
            FP::xacc_mad_(P0, lo0, lo1);
            FP::xacc_mad_(P1, FP::slope(lo0, hi0), FP::slope(lo1, hi1));
        }
        acc[0] = FP::xacc_reduce_(P0); acc[1] = FP::xacc_reduce_(P1);
    } else {
        typename FP::BAcc P0 = FP::bacc_zero(), P1 = FP::bacc_zero(), P2 = FP::bacc_zero();
        for (size_t b = (size_t)blockIdx.x * blockDim.x + threadIdx.x; b < npairs; b += (size_t)gridDim.x * blockDim.x) {
            TIN a[2], c[2];
            load2(in + 2 * b, a);
            load2(in + n_in + 2 * b, c);
            FP::bacc_mad(P0, a[0], c[0]);
            FP::bacc_mad(P1, FP::slope(a[0], a[1]), FP::slope(c[0], c[1]));
            FP::bacc_mad(P2, a[1], c[1]);
        }
        acc[0] = FP::lift(FP::bacc_reduce(P0)); acc[1] = FP::lift(FP::bacc_reduce(P1)); acc[2] = FP::lift(FP::bacc_reduce(P2));
    }
    block_reduce_finalize_ex<FP, NP>(acc, partials, counter, msg, gridDim.x, blockIdx.x);
}

// ---- final folds and captures: out[i] = in[2 i] + r (in[2 i + 1] - in[2 i]) for tiny tables (one item per block)
template <class FP> struct FoldItem {
    const void* in; typename FP::X* out; const typename FP::X* r; int n_out, in_base;
};
template <class FP> __global__ void k_fold_items(const FoldItem<FP>* __restrict__ items) {
    typedef typename FP::B B;
    typedef typename FP::X X;
    const FoldItem<FP> it = items[blockIdx.x];
    const X r = *it.r;
    const typename FP::FoldAux aux = FP::fold_aux(r);
    for (int i = threadIdx.x; i < it.n_out; i += blockDim.x) {
        if (it.in_base) { const B* s = (const B*)it.in; it.out[i] = FP::fold(s[2 * i], s[2 * i + 1], r, aux); }
        else { const X* s = (const X*)it.in; it.out[i] = FP::fold(s[2 * i], s[2 * i + 1], r, aux); }
    }
}
template <class FP> struct CopyItem { const typename FP::X* src; typename FP::X* dst; int n; };
template <class FP> __global__ void k_copy_items(const CopyItem<FP>* __restrict__ items) {
    const CopyItem<FP> it = items[blockIdx.x];
    for (int i = threadIdx.x; i < it.n; i += blockDim.x) it.dst[i] = it.src[i];
}
// constant part of linear layers: out = sum_g W[g] * c[g]
template <class FP>
__global__ void k_dot_wconst(const typename FP::X* __restrict__ w, const typename FP::B* __restrict__ c, size_t n, typename FP::X* partials,
                             unsigned* counter, typename FP::X* out) {
    typedef typename FP::X X;
    typename FP::XAcc a = FP::xacc_zero_();
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) FP::xacc_mad_b(a, w[i], c[i]);
    X acc[1] = {FP::xacc_reduce_(a)};
    block_reduce_finalize<FP, 1>(acc, partials, counter, out);
}

}  // namespace hg
