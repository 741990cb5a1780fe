// Round 0 of the grand-product layer sumchecks, fused into the kernels that BUILD the product trees (prefetch mode).
//
// Reference: /root/reference/lasso/src/memory_checking/prover.rs:223-279 (layer sumcheck), :332-354 (Layer::up).
// Round 0 of the sumcheck on a tree layer samples
//        h(X) = sum_b t_0(b; X) * sum_i c_i * l_i(b; X) * r_i(b; X)
// on the UNFOLDED layer, i.e. on exactly the values the tree builder holds in registers when it multiplies l_i * r_i to
// get the layer above: q_i(b; 0) = l_i(2b) r_i(2b) and q_i(b; 1) = l_i(2b+1) r_i(2b+1) ARE the two tree entries it writes.
// With all challenges known up front (c_i = gamma_layer^i, transcript.rs:156,183-203) the builder therefore emits the four
// samples h(0), h(inf), h(-1), h(1) itself and the layer is never re-read for round 0 (2.6 GB less traffic per proof at
// n = 32768 than a separate round-0 pass).
//   * q_i(b; X) = l_i r_i is quadratic in X: q(inf) costs one product of slopes, q(-1) = 2 q(0) - q(1) + 2 q(inf) none;
//   * per vector i the base-field sums D_i(p) = sum_b t_0(b; p) q_i(b; p) are accumulated unreduced and multiplied by the
//     extension coefficient c_i once per thread;
//   * every CTA writes its four partial sums; the tail kernel of the layer (its first CTA, gp_kernels.cuh) adds them
//     up. Field addition is exact, so the order of summation does not change a bit of the message.
// Blocks are numbered vector-fastest: the CTAs of one position range run back to back and share the t_0 segment (vector 0)
// and, in the hash kernel, the address / counter columns of a chunk through L2.
#pragma once
#include "gp_kernels.cuh"

namespace hg {

constexpr int HG_FUSED_BLOCK = 128;

// block-level sum of NP BASE values; thread 0 ends up with the sums in v[0..NP). The CTAs of these kernels work on one vector
// (two in the hash kernel), so the extension coefficient c_i is applied once per CTA, after this reduction.
template <class FP, int NP> __device__ __forceinline__ void block_sum_base(typename FP::B (&v)[NP]) {
    typedef typename FP::B B;
    __shared__ B red[32][NP];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = (blockDim.x + 31) >> 5;
#pragma unroll
    for (int p = 0; p < NP; p++) {
        B s = v[p];
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) s = FP::b_add(s, FP::b_shfl_down(s, off));
        if (lane == 0) red[warp][p] = s;
    }
    __syncthreads();
    if (warp == 0) {
#pragma unroll
        for (int p = 0; p < NP; p++) {
            B s = lane < nwarps ? red[lane][p] : FP::b_zero();
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) s = FP::b_add(s, FP::b_shfl_down(s, off));
            v[p] = s;
        }
    }
}

// D[0..3] += samples of t_0 * q at X = 0, inf, -1, 1 for one pair position. q0 = l_lo r_lo and q1 = l_hi r_hi are the entries of
// the layer above (canonical); all other inputs canonical.
template <class FP>
__device__ __forceinline__ void r0_accumulate(typename FP::BAcc (&D)[4], const typename FP::B& t_lo, const typename FP::B& t_hi, const typename FP::B& l_lo,
                                              const typename FP::B& l_hi, const typename FP::B& r_lo, const typename FP::B& r_hi, const typename FP::B& q0,
                                              const typename FP::B& q1) {
    typedef typename FP::B B;
    const B qinf = FP::fmul(FP::slope(l_lo, l_hi), FP::slope(r_lo, r_hi));
    const B qm1 = FP::q_at_m1(q0, q1, qinf);  // q(-1) = 2 q(0) - q(1) + 2 q(inf), any representative
    FP::bacc_mad(D[0], t_lo, q0);
    FP::bacc_mad(D[1], FP::slope(t_lo, t_hi), qinf);
    FP::bacc_mad(D[2], FP::at_m1(t_lo, t_hi), qm1);
    FP::bacc_mad(D[3], t_hi, q1);
}

// ---- hash build (prover.rs:35-89) + first tree level + round 0 of the bottom layer.  V = layer 0 ([2m][R]), up = layer 1.
// grid = nxb * m blocks, block b: memory position b % m, position range b / m.  part: [grid][4].
template <class FP>
__global__ void __launch_bounds__(HG_FUSED_BLOCK, FP::FUSED_MIN_BLOCKS)
k_hash_rw_up_r0(const u16* __restrict__ dims, const u32* __restrict__ read_cts, const typename FP::B* __restrict__ E, const int* __restrict__ pos_mem,
                const int* __restrict__ pos_dim, const int* __restrict__ pos_slot, const typename FP::X* __restrict__ gamma_tau, size_t R, int m,
                typename FP::B* __restrict__ V, typename FP::B* __restrict__ up, VecRange own, const typename FP::X* __restrict__ c,
                typename FP::X* __restrict__ part, int nxb) {
    typedef typename FP::B B;
    typedef typename FP::X X;
    const size_t h = R / 2;
    const int pos = blockIdx.x % m, xb = blockIdx.x / m;
    X* my = part + (size_t)blockIdx.x * 4;
    const bool need_r = vec_needed(own, pos), need_w = vec_needed(own, m + pos);
    const bool own_r = pos >= own.lo && pos < own.hi, own_w = m + pos >= own.lo && m + pos < own.hi;
    if (!need_r && !need_w) {
        if (threadIdx.x < 4) my[threadIdx.x] = FP::x_zero();
        return;
    }
    const B gamma = FP::x_base0(gamma_tau[0]), tau = FP::x_base0(gamma_tau[1]), gamma2 = FP::b_mul(gamma, gamma);
    const u16* dm = dims + (size_t)pos_dim[pos] * R;
    const u32* ts = read_cts + (size_t)pos_slot[pos] * R;
    const B* e = E + (size_t)pos_mem[pos] * R;
    const B mtau = FP::b_sub(FP::b_zero(), tau);
    // a + e*gamma + t*gamma^2 - tau with one reduction
    auto hash = [&](size_t q) {
        typename FP::BAcc acc = FP::bacc_zero();
        FP::bacc_mad(acc, e[q], gamma);
        FP::bacc_mad(acc, FP::to_base(ts[q]), gamma2);
        FP::bacc_add(acc, FP::to_base(dm[q]));
        FP::bacc_add(acc, mtau);
        return FP::bacc_reduce(acc);
    };
    B* Vr = V + (size_t)pos * R;
    B* Vw = V + (size_t)(m + pos) * R;
    B* ur = up + (size_t)pos * h;
    B* uw = up + (size_t)(m + pos) * h;
    typename FP::BAcc Dr[4], Dw[4];
#pragma unroll
    for (int p = 0; p < 4; p++) { Dr[p] = FP::bacc_zero(); Dw[p] = FP::bacc_zero(); }
    for (size_t t = (size_t)xb * blockDim.x + threadIdx.x; t < h / 2; t += (size_t)nxb * blockDim.x) {
        const size_t j0 = 2 * t;
        B rd[2][2], wr[2][2];  // [row j0 + u][half s]
#pragma unroll
        for (int u = 0; u < 2; u++)
#pragma unroll
            for (int s = 0; s < 2; s++) {
                rd[u][s] = hash(j0 + u + s * h);
                wr[u][s] = FP::b_add(rd[u][s], gamma2);
            }
        B t0[2];
        if (pos == 0) { t0[0] = rd[0][0]; t0[1] = rd[1][0]; }
        else load_pair(V + j0, t0[0], t0[1]);  // first half of vector 0, written by k_hash_t0 before this launch
        if (need_r) {
            const B q0 = FP::fmul(rd[0][0], rd[0][1]), q1 = FP::fmul(rd[1][0], rd[1][1]);
            if (pos != 0) store_pair(Vr + j0, rd[0][0], rd[1][0]);  // (vector 0's first half is already there and is being read by the other CTAs)
            store_pair(Vr + j0 + h, rd[0][1], rd[1][1]);
            store_pair(ur + j0, q0, q1);
            if (own_r) r0_accumulate<FP>(Dr, t0[0], t0[1], rd[0][0], rd[1][0], rd[0][1], rd[1][1], q0, q1);
        }
        if (need_w) {
            const B q0 = FP::fmul(wr[0][0], wr[0][1]), q1 = FP::fmul(wr[1][0], wr[1][1]);
#pragma unroll
            for (int s = 0; s < 2; s++) store_pair(Vw + j0 + s * h, wr[0][s], wr[1][s]);
            store_pair(uw + j0, q0, q1);
            if (own_w) r0_accumulate<FP>(Dw, t0[0], t0[1], wr[0][0], wr[1][0], wr[0][1], wr[1][1], q0, q1);
        }
    }
    B v[8];
#pragma unroll
    for (int p = 0; p < 4; p++) { v[p] = FP::bacc_reduce(Dr[p]); v[4 + p] = FP::bacc_reduce(Dw[p]); }
    block_sum_base<FP, 8>(v);
    if (threadIdx.x == 0) {
        const X cr = c[pos], cw = c[m + pos];
#pragma unroll
        for (int p = 0; p < 4; p++) {
            typename FP::XAcc a = FP::xacc_zero_();
            if (own_r) FP::xacc_mad_b(a, cr, v[p]);
            if (own_w) FP::xacc_mad_b(a, cw, v[4 + p]);
            my[p] = FP::xacc_reduce_(a);
        }
    }
}

// first half of vector 0 of the bottom layer (= t_0 of its sumcheck), computed before k_hash_rw_up_r0 so that every CTA of that
// launch can read it instead of hashing memory 0 again
template <class FP>
__global__ void k_hash_t0(const u16* __restrict__ dims, const u32* __restrict__ read_cts, const typename FP::B* __restrict__ E, const int* __restrict__ pos_mem,
                          const int* __restrict__ pos_dim, const int* __restrict__ pos_slot, const typename FP::X* __restrict__ gamma_tau, size_t R,
                          typename FP::B* __restrict__ V) {
    typedef typename FP::B B;
    const size_t j0 = 2 * ((size_t)blockIdx.x * blockDim.x + threadIdx.x);
    if (j0 >= R / 2) return;
    const B gamma = FP::x_base0(gamma_tau[0]), tau = FP::x_base0(gamma_tau[1]), gamma2 = FP::b_mul(gamma, gamma), mtau = FP::b_sub(FP::b_zero(), tau);
    const u16* dm = dims + (size_t)pos_dim[0] * R;
    const u32* ts = read_cts + (size_t)pos_slot[0] * R;
    const B* e = E + (size_t)pos_mem[0] * R;
    B o[2];
#pragma unroll
    for (int u = 0; u < 2; u++) {
        typename FP::BAcc acc = FP::bacc_zero();
        FP::bacc_mad(acc, e[j0 + u], gamma);
        FP::bacc_mad(acc, FP::to_base(ts[j0 + u]), gamma2);
        FP::bacc_add(acc, FP::to_base(dm[j0 + u]));
        FP::bacc_add(acc, mtau);
        o[u] = FP::bacc_reduce(acc);
    }
    store_pair(V + j0, o[0], o[1]);
}

// ---- product-tree levels (prover.rs:332-354) + round 0 of the layers they touch.
//   TWO:  in = layer k-1 [nvec][4q] -> out1 = layer k [nvec][2q] -> out2 = layer k+1 [nvec][q]; round 0 of layers k-1 (partA) and k (partB)
//   !TWO: in = layer k-1 [nvec][2q] -> out1 = layer k [nvec][q];                                round 0 of layer k-1 (partA)
// grid = nxb * nvec blocks, block b: vector b % nvec, position range b / nvec.  q >= 2.
template <class FP> struct TreeR0Args {
    const typename FP::B* in;
    typename FP::B* out1;
    typename FP::B* out2;
    const typename FP::X* cA;
    const typename FP::X* cB;
    typename FP::X* partA;
    typename FP::X* partB;
    unsigned long long q;
    int nvec, nxb;
    VecRange own;
};
// The two product trees of a node (read / write sets over R rows, init / final sets over M entries) are independent: step k of both
// goes into ONE launch (blocks [0, nblk_a) work for tree a, the rest for tree b), so the short launches of the small tree disappear
// into those of the large one (nblk_a = gridDim.x: a single tree).
template <class FP, bool TWO>
__global__ void __launch_bounds__(HG_FUSED_BLOCK, FP::FUSED_MIN_BLOCKS) k_tree_up_r0(const TreeR0Args<FP> a_first, const TreeR0Args<FP> a_second, unsigned nblk_a) {
    typedef typename FP::B B;
    typedef typename FP::X X;
    const bool second = blockIdx.x >= nblk_a;
    const TreeR0Args<FP>& a = second ? a_second : a_first;
    const unsigned bid = blockIdx.x - (second ? nblk_a : 0u);
    const int i = bid % a.nvec, xb = bid / a.nvec;
    const size_t q = a.q;
    X* myA = a.partA + (size_t)bid * 4;
    X* myB = TWO ? a.partB + (size_t)bid * 4 : nullptr;
    if (!vec_needed(a.own, i)) {
        if (threadIdx.x < 4) { myA[threadIdx.x] = FP::x_zero(); if (TWO) myB[threadIdx.x] = FP::x_zero(); }
        return;
    }
    const bool owned = i >= a.own.lo && i < a.own.hi;
    constexpr int NQ = TWO ? 4 : 2;
    const B* v = a.in + (size_t)i * NQ * q;
    const B* v0 = a.in;  // vector 0: its first half is t_0
    B* o1 = a.out1 + (size_t)i * (NQ / 2) * q;
    B* o2 = TWO ? a.out2 + (size_t)i * q : nullptr;
    typename FP::BAcc DA[4], DB[4];
#pragma unroll
    for (int p = 0; p < 4; p++) { DA[p] = FP::bacc_zero(); DB[p] = FP::bacc_zero(); }
    for (size_t t = (size_t)xb * blockDim.x + threadIdx.x; t < q / 2; t += (size_t)a.nxb * blockDim.x) {
        const size_t k = 2 * t;
        B x[NQ][2];
#pragma unroll
        for (int s = 0; s < NQ; s++) load_pair(v + k + s * q, x[s][0], x[s][1]);
        if constexpr (TWO) {
            // layer k-1: l = quarters 0, 1; r = quarters 2, 3.  layer k: l' = a (positions k..), r' = b (positions k + q..)
            B pa[2], pb[2], po[2];
#pragma unroll
            for (int u = 0; u < 2; u++) { pa[u] = FP::fmul(x[0][u], x[2][u]); pb[u] = FP::fmul(x[1][u], x[3][u]); po[u] = FP::fmul(pa[u], pb[u]); }
            store_pair(o1 + k, pa[0], pa[1]);
            store_pair(o1 + k + q, pb[0], pb[1]);
            store_pair(o2 + k, po[0], po[1]);
            if (owned) {
                B t0[2][2], ta[2];
                if (i == 0) {
#pragma unroll
                    for (int u = 0; u < 2; u++) { t0[0][u] = x[0][u]; t0[1][u] = x[1][u]; ta[u] = pa[u]; }
                } else {
                    B t2[2];
                    load_pair(v0 + k, t0[0][0], t0[0][1]);
                    load_pair(v0 + k + q, t0[1][0], t0[1][1]);
                    load_pair(v0 + k + 2 * q, t2[0], t2[1]);
#pragma unroll
                    for (int u = 0; u < 2; u++) ta[u] = FP::fmul(t0[0][u], t2[u]);
                }
                r0_accumulate<FP>(DA, t0[0][0], t0[0][1], x[0][0], x[0][1], x[2][0], x[2][1], pa[0], pa[1]);
                r0_accumulate<FP>(DA, t0[1][0], t0[1][1], x[1][0], x[1][1], x[3][0], x[3][1], pb[0], pb[1]);
                r0_accumulate<FP>(DB, ta[0], ta[1], pa[0], pa[1], pb[0], pb[1], po[0], po[1]);
            }
        } else {
            B pa[2];
#pragma unroll
            for (int u = 0; u < 2; u++) pa[u] = FP::fmul(x[0][u], x[1][u]);
            store_pair(o1 + k, pa[0], pa[1]);
            if (owned) {
                B t0[2];
                if (i == 0) { t0[0] = x[0][0]; t0[1] = x[0][1]; }
                else load_pair(v0 + k, t0[0], t0[1]);
                r0_accumulate<FP>(DA, t0[0], t0[1], x[0][0], x[0][1], x[1][0], x[1][1], pa[0], pa[1]);
            }
        }
    }
    constexpr int NP = TWO ? 8 : 4;
    B vv[NP];
#pragma unroll
    for (int p = 0; p < 4; p++) vv[p] = FP::bacc_reduce(DA[p]);
    if constexpr (TWO) {
#pragma unroll
        for (int p = 0; p < 4; p++) vv[4 + p] = FP::bacc_reduce(DB[p]);
    }
    block_sum_base<FP, NP>(vv);
    if (threadIdx.x == 0) {
        const X ca = a.cA[i];
#pragma unroll
        for (int p = 0; p < 4; p++) myA[p] = owned ? FP::fmul_any(ca, vv[p]) : FP::x_zero();
        if constexpr (TWO) {
            const X cb = a.cB[i];
#pragma unroll
            for (int p = 0; p < 4; p++) myB[p] = owned ? FP::fmul_any(cb, vv[4 + p]) : FP::x_zero();
        }
    }
}

}  // namespace hg
