// Batched verification of GKR proofs on the device (hg_verifier_new / hg_gkr_verify_batch / hg_mle_eval_multi).
//
// A batch is B proofs of one circuit. Each proof is replayed on the host by GkrVerifierHost::verify with a DeferredChecks sink
// (gkr_verify.hpp): every transcript operation and every scalar check runs there, and the final checks whose quantity is linear
// in the circuit size are left as records sum_j coef[j] * q[j] == target (lasso_verify.hpp). This file computes the q of all
// records of the batch on the device and closes them:
//   DC_FFT       W = sum_t alpha^t eq(z_t, .) (k_eq_split_multi + k_eq_accumulate), transform(W) (k_ext_split + NTT + k_ext_merge),
//                then transform(W) . eq(pt) (k_dot_eq_items over the extension table)
//   DC_LINEAR    W as above, then one pass over the node's additive edges and constants (k_edge_sum)
//   DC_GENERAL   W as above, A(u) and the constant part as for DC_LINEAR at pt = u, then one pass over the node's product edges
//                with eq(u, .) and eq(v, .) (k_mul_edge_sum)
//   DC_SUBTABLE  subtable . eq(y), the subtables uploaded once by the verifier
//   DC_INPUT     input table . eq(pt), for every (proof, input, claim)
// Every stage is one launch over all items. A quantity is keyed by the bytes of what determines it (node, claim points, alpha,
// point, a general layer's v; for inputs also the table), so proofs that carry the same points, as every proof of the library's
// Keccak256Transcript does, share one W, one transform, one dot and one edge sum. Proofs with their own points get their own
// (processed in groups that fit the weight pool).
#pragma once
#include <array>
#include <chrono>
#include <cstring>
#include <map>
#include <string>

#include "gkr_verify.hpp"
#include "ntt_engine.cuh"

namespace hg {

// out = sum_i eq(pt, i) t[i] for one item, eq(pt, .) in two factors: eq_lo over the low lo_bits variables, eq_hi over the rest.
// Blocks blk_start .. blk_start + nblk - 1 belong to the item; each reduces rows of 2^lo_bits entries.
template <class FP, class T> struct DotItem {
    const T* t;
    const typename FP::X* eq_lo;
    const typename FP::X* eq_hi;
    typename FP::X* out;
    typename FP::X* partials;
    unsigned* counter;
    u64 n;
    int lo_bits, blk_start, nblk;
};
template <class FP, class T> __global__ void __launch_bounds__(HG_BLOCK) k_dot_eq_items(const DotItem<FP, T>* __restrict__ items, int nitems) {
    typedef typename FP::X X;
    const DotItem<FP, T> it = items[find_item(items, nitems)];
    const unsigned bid = blockIdx.x - it.blk_start;
    const size_t nlo = (size_t)1 << it.lo_bits, nhi = it.n >> it.lo_bits;
    X acc[1] = {FP::x_zero()};
    for (size_t kh = bid; kh < nhi; kh += it.nblk) {
        const T* row = it.t + kh * nlo;
        X a = FP::x_zero();
        for (size_t kl = threadIdx.x; kl < nlo; kl += blockDim.x) a = FP::x_add(a, FP::mul(it.eq_lo[kl], row[kl]));
        acc[0] = FP::x_add(acc[0], FP::mul(a, it.eq_hi[kh]));
    }
    block_reduce_finalize_ex<FP, 1>(acc, it.partials, it.counter, it.out, (unsigned)it.nblk, bid);
}

// A linear layer's deferred quantities in one pass over its edges: out[0] = sum_e coef_e W[out_e] eq(pt, in_e) = MLE(A)(pt),
// out[1] = sum over the constant gates of const_g W[g] (entries with in_e == HG_EDGE_CONST)
constexpr u32 HG_EDGE_CONST = 0xffffffffu;
template <class FP> struct EdgeItem {
    const u32* out_idx;
    const u32* in_idx;
    const typename FP::B* coef;
    const typename FP::X* w;
    const typename FP::X* eq_lo;
    const typename FP::X* eq_hi;
    typename FP::X* out;
    typename FP::X* partials;
    unsigned* counter;
    u64 n;
    int lo_bits, blk_start, nblk;
};
template <class FP> __global__ void __launch_bounds__(HG_BLOCK) k_edge_sum(const EdgeItem<FP>* __restrict__ items, int nitems) {
    typedef typename FP::X X;
    const EdgeItem<FP> it = items[find_item(items, nitems)];
    const unsigned bid = blockIdx.x - it.blk_start;
    const u32 lo_mask = (1u << it.lo_bits) - 1;
    X acc[2] = {FP::x_zero(), FP::x_zero()};
    for (size_t e = (size_t)bid * blockDim.x + threadIdx.x; e < it.n; e += (size_t)it.nblk * blockDim.x) {
        const X wc = FP::mul(it.w[it.out_idx[e]], it.coef[e]);
        const u32 in = it.in_idx[e];
        if (in == HG_EDGE_CONST) acc[1] = FP::x_add(acc[1], wc);
        else acc[0] = FP::x_add(acc[0], FP::mul(wc, FP::mul(it.eq_lo[in & lo_mask], it.eq_hi[in >> it.lo_bits])));
    }
    block_reduce_finalize_ex<FP, 2>(acc, it.partials, it.counter, it.out, (unsigned)it.nblk, bid);
}

// A general layer's product part in one pass over its product edges: out[0] = sum_e coef_e W[out_e] eq(u, x_e) eq(v, y_e) = M(u, v),
// with x_e, y_e the two factors' positions in the concatenated inputs (num_reps expanded) and eq(u, .), eq(v, .) in two factors each
template <class FP> struct MulEdgeItem {
    const u32* out_idx;
    const u32* x_idx;
    const u32* y_idx;
    const typename FP::B* coef;
    const typename FP::X* w;
    const typename FP::X* equ_lo;
    const typename FP::X* equ_hi;
    const typename FP::X* eqv_lo;
    const typename FP::X* eqv_hi;
    typename FP::X* out;
    typename FP::X* partials;
    unsigned* counter;
    u64 n;
    int lo_bits, blk_start, nblk;
};
template <class FP> __global__ void __launch_bounds__(HG_BLOCK) k_mul_edge_sum(const MulEdgeItem<FP>* __restrict__ items, int nitems) {
    typedef typename FP::X X;
    const MulEdgeItem<FP> it = items[find_item(items, nitems)];
    const unsigned bid = blockIdx.x - it.blk_start;
    const u32 lo_mask = (1u << it.lo_bits) - 1;
    X acc[1] = {FP::x_zero()};
    for (size_t e = (size_t)bid * blockDim.x + threadIdx.x; e < it.n; e += (size_t)it.nblk * blockDim.x) {
        const u32 x = it.x_idx[e], y = it.y_idx[e];
        const X wc = FP::mul(it.w[it.out_idx[e]], it.coef[e]);
        const X eu = FP::mul(it.equ_lo[x & lo_mask], it.equ_hi[x >> it.lo_bits]), ev = FP::mul(it.eqv_lo[y & lo_mask], it.eqv_hi[y >> it.lo_bits]);
        acc[0] = FP::x_add(acc[0], FP::mul(wc, FP::mul(eu, ev)));
    }
    block_reduce_finalize_ex<FP, 1>(acc, it.partials, it.counter, it.out, (unsigned)it.nblk, bid);
}

// Device scratch shared by the stages: descriptor staging through one pinned arena, eq factor pool, partial sums and counters.
// Everything staged is valid until finish() synchronises the stream.
template <class FP> class VerifyScratch {
  public:
    typedef typename FP::X X;
    explicit VerifyScratch(DeviceCtx* ctx) : ctx_(ctx) {}
    template <class T> const T* stage(const std::vector<T>& v) {
        const size_t bytes = (v.size() * sizeof(T) + 15) & ~(size_t)15;
        if (off_ + bytes > h_.n) throw std::runtime_error("verify: descriptor staging overflow");
        memcpy(h_.p + off_, v.data(), v.size() * sizeof(T));
        HG_CUDA(cudaMemcpyAsync(d_.p + off_, h_.p + off_, bytes, cudaMemcpyHostToDevice, ctx_->stream));
        const T* r = (const T*)(d_.p + off_);
        off_ += bytes;
        return r;
    }
    // sizes every pool for one round of at most `items` reductions (three output slots each), `blocks` reduction blocks (two sums
    // each), `eq` eq-factor entries and `desc` descriptor bytes; waits for the stream before it replaces a buffer
    void reserve(size_t items, size_t blocks, size_t eq, size_t desc) {
        auto grow = [&](auto& b, size_t need) { if (b.n < need) { HG_CUDA(cudaStreamSynchronize(ctx_->stream)); b.alloc(need + need / 2); } };
        grow(out, 3 * items);
        grow(partials, 2 * blocks);
        grow(eq_pool, eq);
        if (counters.n < items) {
            grow(counters, items);
            HG_CUDA(cudaMemsetAsync(counters.p, 0, counters.bytes(), ctx_->stream));  // each reduction leaves its counter at 0
        }
        if (h_.n < desc) { HG_CUDA(cudaStreamSynchronize(ctx_->stream)); h_.alloc(2 * desc); d_.alloc(2 * desc); off_ = 0; }
        if (h_out.n < out.n) h_out.alloc(out.n);
    }
    // downloads the first n_out outputs and resets the staging arena
    void finish(size_t n_out) {
        if (n_out) HG_CUDA(cudaMemcpyAsync(h_out.p, out.p, n_out * sizeof(X), cudaMemcpyDeviceToHost, ctx_->stream));
        HG_CUDA(cudaStreamSynchronize(ctx_->stream));
        off_ = 0;
    }
    DevBuf<X> out, partials, eq_pool;
    DevBuf<unsigned> counters;
    PinnedBuf<X> h_out;

  private:
    DeviceCtx* ctx_;
    PinnedBuf<unsigned char> h_;
    DevBuf<unsigned char> d_;
    size_t off_ = 0;
};

// Base-table MLEs at per-item points (hg_mle_eval_multi, the verifier's subtables and input claims): one eq-factor launch for the
// distinct points, one dot launch for all items. Returns the values in item order.
template <class FP> std::vector<typename FP::X> mle_eval_items(DeviceCtx* ctx, VerifyScratch<FP>& sc, const std::vector<const typename FP::B*>& tables,
                                                             const std::vector<const std::vector<typename FP::X>*>& points) {
    typedef typename FP::X X;
    typedef typename FP::B B;
    const size_t n = tables.size();
    std::vector<X> res(n);
    if (!n) return res;
    // distinct points, each with its eq factors in the pool
    std::map<std::string, size_t> seen;
    std::vector<size_t> pt_of(n), eq_off;
    std::vector<const std::vector<X>*> pts;
    size_t eq_need = 0, blocks = 0;
    auto lo_of = [](size_t nv) { return (int)std::min<size_t>(nv, 10); };
    for (size_t i = 0; i < n; i++) {
        const std::vector<X>& p = *points[i];
        std::string key((const char*)p.data(), p.size() * sizeof(X));
        auto it = seen.find(key);
        if (it == seen.end()) {
            it = seen.emplace(key, pts.size()).first;
            pts.push_back(&p);
            eq_off.push_back(eq_need);
            const int lo = lo_of(p.size());
            eq_need += ((size_t)1 << lo) + ((size_t)1 << (p.size() - lo));
        }
        pt_of[i] = it->second;
        const int lo = lo_of(p.size());
        blocks += std::min<size_t>((size_t)1 << (p.size() - lo), 16);
    }
    size_t pt_elems = 0;
    for (auto* p : pts) pt_elems += p->size();
    sc.reserve(n, blocks, eq_need, pts.size() * sizeof(EqSplitItem<FP>) + n * sizeof(DotItem<FP, B>) + pt_elems * sizeof(X) + 1024);
    std::vector<X> flat(1, FP::x_zero());  // never empty: a table of one entry has a point of no coordinates
    for (auto* p : pts) flat.insert(flat.end(), p->begin(), p->end());
    const X* d_pts = sc.stage(flat) + 1;
    std::vector<EqSplitItem<FP>> splits;
    int split_blk = 0;
    size_t poff = 0;
    for (size_t k = 0; k < pts.size(); k++) {
        const int nv = (int)pts[k]->size(), lo = lo_of(nv);
        EqSplitItem<FP> si;
        si.point = d_pts + poff; si.eq_lo = sc.eq_pool.p + eq_off[k]; si.eq_hi = si.eq_lo + ((size_t)1 << lo); si.alpha = nullptr;
        si.nv = nv; si.lo_bits = lo; si.blk_start = split_blk; si.t = 0;
        split_blk += (int)((((size_t)1 << lo) + ((size_t)1 << (nv - lo)) + HG_BLOCK - 1) / HG_BLOCK);
        splits.push_back(si);
        poff += nv;
    }
    HG_K(ctx, KC_GKR_PREP, eq_need * sizeof(X), k_eq_split_multi<FP><<<split_blk, HG_BLOCK, 0, ctx->stream>>>(sc.stage(splits), (int)splits.size()));
    std::vector<DotItem<FP, B>> items;
    int blk = 0;
    size_t bytes = 0, pblk = 0;
    for (size_t i = 0; i < n; i++) {
        const EqSplitItem<FP>& si = splits[pt_of[i]];
        DotItem<FP, B> d;
        d.t = tables[i]; d.eq_lo = si.eq_lo; d.eq_hi = si.eq_hi; d.out = sc.out.p + i; d.partials = sc.partials.p + pblk; d.counter = sc.counters.p + i;
        d.n = (u64)1 << si.nv; d.lo_bits = si.lo_bits; d.blk_start = blk; d.nblk = (int)std::min<size_t>((size_t)1 << (si.nv - si.lo_bits), 16);
        blk += d.nblk;
        pblk += d.nblk;
        bytes += d.n * sizeof(B);
        items.push_back(d);
    }
    HG_K(ctx, KC_DOT, bytes, k_dot_eq_items<FP, B><<<blk, HG_BLOCK, 0, ctx->stream>>>(sc.stage(items), (int)items.size()));
    sc.finish(n);
    for (size_t i = 0; i < n; i++) res[i] = sc.h_out.p[i];
    return res;
}

template <class FP> class VerifierDev {
  public:
    typedef typename FP::B B;
    typedef typename FP::X X;
    typedef typename GkrVerifierHost<FP>::Claim Claim;
    struct Result { bool ok = true; std::string reason; };

    VerifierDev(DeviceCtx* ctx, NttEngine<FP>* ntt, const GkrVerifierHost<FP>& desc, size_t max_batch)
        : ctx_(ctx), ntt_(ntt), desc_(desc), max_batch_(max_batch), sc_(ctx) {
        if (max_batch < 1) throw std::runtime_error("hg_verifier_new: max_batch must be at least 1");
        input_lens_ = desc.input_lens();
        size_t w_total = 0;
        const LassoPreprocessing* pp = nullptr;
        for (int id = 0; id < (int)desc.num_nodes(); id++) {
            if (desc.node_kind(id) == GKR_LASSO) {
                if (pp) throw std::runtime_error("hg_verifier_new: the device verifier takes at most one Lasso node");
                pp = desc.node_lasso(id);
            }
            if (desc.node_kind(id) == GKR_FFT) w_total += desc.node_out_len(id);
            const bool general = desc.node_is_general(id);
            if (!desc.node_is_linear(id) && !general) continue;
            w_total += desc.node_out_len(id);
            // the additive edges as (output, concatenated input, coefficient), constants as (gate, HG_EDGE_CONST, const)
            const VanillaDesc& d = *desc.node_desc(id);
            const size_t ng = desc.node_num_gates(id), n_in = desc.node_n_in(id), sub = (size_t)1 << d.log2_sub;
            if (desc.node_in_len(id) > HG_EDGE_CONST || desc.node_out_len(id) > HG_EDGE_CONST) throw std::runtime_error("hg_verifier_new: layer too large");
            std::vector<u32> out_idx, in_idx, mul_out, mul_x, mul_y;
            std::vector<B> coef, mul_coef;
            for (size_t r = 0; r < (size_t)desc.node_num_reps(id); r++)
                for (size_t g = 0; g < ng; g++) {
                    const u32 o = (u32)(r * ng + g);
                    if (d.has_const[g]) { out_idx.push_back(o); in_idx.push_back(HG_EDGE_CONST); coef.push_back(FP::b_from_limbs(&d.consts[g * FP::B_LIMBS])); }
                    for (uint64_t e = d.add_ptr[g]; e < d.add_ptr[g + 1]; e++) {
                        out_idx.push_back(o);
                        in_idx.push_back((u32)((size_t)d.add_in[e] * n_in + r * sub + d.add_wire[e]));
                        coef.push_back(FP::b_from_limbs(&d.add_coef[e * FP::B_LIMBS]));
                    }
                    // general layers: the product edges as (output, x, y, coefficient)
                    for (uint64_t e = d.mul_ptr[g]; general && e < d.mul_ptr[g + 1]; e++) {
                        mul_out.push_back(o);
                        mul_x.push_back((u32)((size_t)d.mul_in0[e] * n_in + r * sub + d.mul_w0[e]));
                        mul_y.push_back((u32)((size_t)d.mul_in1[e] * n_in + r * sub + d.mul_w1[e]));
                        mul_coef.push_back(FP::b_from_limbs(&d.mul_coef[e * FP::B_LIMBS]));
                    }
                }
            Edges& E = edges_[id];
            E.n = out_idx.size();
            E.out_idx.alloc(std::max<size_t>(E.n, 1)); E.in_idx.alloc(std::max<size_t>(E.n, 1)); E.coef.alloc(std::max<size_t>(E.n, 1));
            upload(E.out_idx.p, out_idx); upload(E.in_idx.p, in_idx); upload(E.coef.p, coef);
            if (!general) continue;
            MulEdges& M = mul_edges_[id];
            M.n = mul_out.size();
            M.out_idx.alloc(std::max<size_t>(M.n, 1)); M.x_idx.alloc(std::max<size_t>(M.n, 1)); M.y_idx.alloc(std::max<size_t>(M.n, 1));
            M.coef.alloc(std::max<size_t>(M.n, 1));
            upload(M.out_idx.p, mul_out); upload(M.x_idx.p, mul_x); upload(M.y_idx.p, mul_y); upload(M.coef.p, mul_coef);
        }
        if (pp) {  // every subtable, materialised once
            const size_t M = pp->M;
            subtables_.alloc(pp->subtables_by_idx.size() * M);
            std::vector<B> t(M);
            for (size_t s = 0; s < pp->subtables_by_idx.size(); s++) {
                const std::vector<uint64_t> v = pp->subtables_by_idx[s]->materialize(M);
                for (size_t i = 0; i < M; i++) t[i] = FP::b_from_u64(v[i]);
                upload(subtables_.p + s * M, t);
            }
            subtable_len_ = M;
        }
        // weights of up to max_batch proofs with their own points at once (one launch per stage for all of them), within a budget
        const size_t w_set = std::max<size_t>(w_total, 1), budget = ((size_t)4 << 30) / sizeof(X);
        w_pool_.alloc(w_set * std::max<size_t>(1, std::min(max_batch, budget / w_set)));
    }

    size_t max_batch() const { return max_batch_; }
    // host microseconds of the last batch: [replays, device stages (enqueue and wait), closing the records]
    const double* timing() const { return timing_us_; }
    size_t num_inputs() const { return input_lens_.size(); }
    const std::vector<size_t>& input_lens() const { return input_lens_; }

    // inputs[p * num_inputs() + i]: input i of proof p in the library's representation, on the device
    std::vector<Result> verify(const std::vector<Keccak256Transcript<FP>*>& trs, const std::vector<std::vector<Claim>>& output_claims,
                               const std::vector<const B*>& inputs, const WireOptions& wo) {
        const size_t np = trs.size();
        if (np > max_batch_) throw std::runtime_error("hg_gkr_verify_batch: more proofs than the verifier's max_batch");
        std::vector<Result> res(np);
        std::vector<DeferredChecks<FP>> checks(np);
        typedef std::chrono::steady_clock Clock;
        auto us = [](Clock::time_point a, Clock::time_point b) { return std::chrono::duration<double, std::micro>(b - a).count(); };
        const Clock::time_point t0 = Clock::now();
        for (size_t p = 0; p < np; p++) {
            try {
                const std::vector<std::vector<Claim>> ic = desc_.verify(*trs[p], wo, output_claims[p], &checks[p]);
                for (size_t i = 0; i < ic.size(); i++)
                    for (const Claim& c : ic[i]) {
                        if (((size_t)1 << c.point.size()) != input_lens_[i]) throw VerifyError("verify: input claim point does not match the input's size");
                        DeferredCheck<FP> d;
                        d.kind = DC_INPUT; d.index = (int)(p * input_lens_.size() + i); d.pt = c.point;
                        d.coef[0] = FP::x_one(); d.target = c.value;
                        d.what = "verify: input claim does not match the input";
                        checks[p].push_back(std::move(d));
                    }
            } catch (const CudaError&) {
                throw;
            } catch (const std::exception& e) {
                res[p].ok = false; res[p].reason = e.what();
                checks[p].clear();
            }
        }
        const Clock::time_point t1 = Clock::now();
        // the distinct quantities of the batch
        std::map<std::string, size_t> key_to_q;
        std::vector<const DeferredCheck<FP>*> qs;      // first record of each quantity
        std::vector<std::vector<size_t>> q_of(np);
        for (size_t p = 0; p < np; p++)
            for (const DeferredCheck<FP>& d : checks[p]) {
                std::string key((const char*)&d.kind, sizeof d.kind);
                const int idx = d.kind == DC_INPUT ? 0 : d.index;
                key.append((const char*)&idx, sizeof idx);
                if (d.kind == DC_INPUT) { const B* t = inputs.at(d.index); key.append((const char*)&t, sizeof t); }
                if (weighted(d.kind)) {
                    key.append((const char*)&d.alpha, sizeof(X));
                    for (auto& z : d.z) { const size_t k = z.size(); key.append((const char*)&k, sizeof k); key.append((const char*)z.data(), k * sizeof(X)); }
                }
                key.append((const char*)d.pt.data(), d.pt.size() * sizeof(X));
                key.append((const char*)d.v.data(), d.v.size() * sizeof(X));  // a general layer's v is as long as its pt: the key stays unambiguous
                auto it = key_to_q.find(key);
                if (it == key_to_q.end()) { it = key_to_q.emplace(std::move(key), qs.size()).first; qs.push_back(&d); }
                q_of[p].push_back(it->second);
            }
        std::vector<Q> q(qs.size(), Q{FP::x_zero(), FP::x_zero(), FP::x_zero()});
        // table quantities: subtables and inputs
        {
            std::vector<const B*> tabs;
            std::vector<const std::vector<X>*> pts;
            std::vector<size_t> which;
            for (size_t k = 0; k < qs.size(); k++) {
                const DeferredCheck<FP>& d = *qs[k];
                if (d.kind == DC_SUBTABLE) {
                    if (((size_t)1 << d.pt.size()) != subtable_len_) throw std::runtime_error("verify: subtable point does not match the subtable size");
                    tabs.push_back(subtables_.p + (size_t)d.index * subtable_len_);
                } else if (d.kind == DC_INPUT) {
                    tabs.push_back(inputs.at(d.index));
                } else continue;
                pts.push_back(&d.pt);
                which.push_back(k);
            }
            const std::vector<X> v = mle_eval_items<FP>(ctx_, sc_, tabs, pts);
            for (size_t i = 0; i < which.size(); i++) q[which[i]][0] = v[i];
        }
        // weighted quantities, in groups whose weight tables fit the pool
        std::vector<size_t> group;
        size_t used = 0;
        for (size_t k = 0; k < qs.size(); k++) {
            if (!weighted(qs[k]->kind)) continue;
            const size_t need = desc_.node_out_len(qs[k]->index);
            if (used + need > w_pool_.n) { run_weighted(qs, group, q); group.clear(); used = 0; }
            group.push_back(k);
            used += need;
        }
        if (!group.empty()) run_weighted(qs, group, q);
        const Clock::time_point t2 = Clock::now();
        // close every record
        for (size_t p = 0; p < np; p++) {
            if (!res[p].ok) continue;
            for (size_t r = 0; r < checks[p].size(); r++) {
                const DeferredCheck<FP>& d = checks[p][r];
                const size_t k = q_of[p][r];
                X lhs = FP::x_zero();
                for (int j = 0; j < 3; j++) lhs = FP::x_add(lhs, FP::x_mul(d.coef[j], q[k][j]));
                if (!FP::x_eq(lhs, d.target)) { res[p].ok = false; res[p].reason = d.what; break; }
            }
        }
        timing_us_[0] = us(t0, t1); timing_us_[1] = us(t1, t2); timing_us_[2] = us(t2, Clock::now());
        return res;
    }

  private:
    typedef std::array<X, 3> Q;  // the q[j] of one quantity
    struct Edges { DevBuf<u32> out_idx, in_idx; DevBuf<B> coef; size_t n = 0; };
    struct MulEdges { DevBuf<u32> out_idx, x_idx, y_idx; DevBuf<B> coef; size_t n = 0; };
    static bool weighted(int kind) { return kind == DC_FFT || kind == DC_LINEAR || kind == DC_GENERAL; }
    static int eq_lo_bits(size_t nv) { return (int)std::min<size_t>(nv, 12); }
    template <class T> void upload(T* dst, const std::vector<T>& v) {
        if (v.empty()) return;
        HG_CUDA(cudaMemcpyAsync(dst, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice, ctx_->stream));
        HG_CUDA(cudaStreamSynchronize(ctx_->stream));  // v is the caller's temporary
    }

    // W of every quantity in `group`, the FFT transforms, then the dots (FFT), edge sums (linear, general) and product-edge sums
    // (general); quantity g's results go to output slots 3g .. 3g + 2, its q[0 .. 2]
    void run_weighted(const std::vector<const DeferredCheck<FP>*>& qs, const std::vector<size_t>& group, std::vector<Q>& q) {
        cudaStream_t s = ctx_->stream;
        // eq factors: per quantity, the claim factors back to back (stride nlo + nhi), then the factors of pt (and of v)
        size_t eq_need = 0, pt_elems = 0, blocks = 0, n_splits = 0;
        for (size_t k : group) {
            const DeferredCheck<FP>& d = *qs[k];
            const size_t nvw = d.z.at(0).size(), lo = eq_lo_bits(nvw), nv = d.pt.size(), lp = eq_lo_bits(nv), npts = d.v.empty() ? 1 : 2;
            eq_need += d.z.size() * (((size_t)1 << lo) + ((size_t)1 << (nvw - lo))) + npts * (((size_t)1 << lp) + ((size_t)1 << (nv - lp)));
            pt_elems += d.z.size() * nvw + npts * nv + 1;
            n_splits += d.z.size() + npts;
            blocks += 2 * npts * (size_t)ctx_->sm_count;
        }
        sc_.reserve(group.size(), blocks, eq_need,
                    n_splits * sizeof(EqSplitItem<FP>) +
                        group.size() * (sizeof(EqAccItem<FP>) + sizeof(EdgeItem<FP>) + sizeof(MulEdgeItem<FP>) + sizeof(DotItem<FP, X>) + 2 * sizeof(X*)) +
                        pt_elems * sizeof(X) + 4096);
        std::vector<X> flat;  // alphas and points, staged once all items know their offsets
        const X* d_pts = nullptr;
        std::vector<EqSplitItem<FP>> splits;
        std::vector<EqAccItem<FP>> accs;
        struct Ref { X* w; X* plo; X* phi; X* vlo; X* vhi; int lp; };
        std::vector<Ref> refs;
        size_t eoff = 0, woff = 0;
        int split_blk = 0, acc_blk = 0;
        std::vector<std::pair<size_t, size_t>> offs;  // per split: offsets of its point and its alpha (npos: none) in `flat`
        auto split = [&](size_t pt_off, int nv, int lo, size_t alpha_off, int t) {
            EqSplitItem<FP> si;
            offs.push_back({pt_off, alpha_off});
            si.point = nullptr; si.eq_lo = sc_.eq_pool.p + eoff; si.eq_hi = si.eq_lo + ((size_t)1 << lo); si.alpha = nullptr;
            si.nv = nv; si.lo_bits = lo; si.blk_start = split_blk; si.t = t;
            const size_t len = ((size_t)1 << lo) + ((size_t)1 << (nv - lo));
            split_blk += (int)((len + HG_BLOCK - 1) / HG_BLOCK);
            eoff += len;
            splits.push_back(si);
            return si;
        };
        for (size_t k : group) {
            const DeferredCheck<FP>& d = *qs[k];
            const size_t out_len = desc_.node_out_len(d.index);
            const int nvw = (int)d.z[0].size(), lo = eq_lo_bits(nvw);
            const size_t alpha_off = flat.size();
            flat.push_back(d.alpha);
            const size_t a_off = d.z.size() > 1 ? alpha_off : std::string::npos;
            EqAccItem<FP> ai;
            for (size_t t = 0; t < d.z.size(); t++) {
                const size_t off = flat.size();
                flat.insert(flat.end(), d.z[t].begin(), d.z[t].end());
                const EqSplitItem<FP> si = split(off, nvw, lo, a_off, (int)t);
                if (t == 0) ai.eq0 = si.eq_lo;
            }
            ai.w = w_pool_.p + woff; ai.n = out_len; ai.stride = ((size_t)1 << lo) + (out_len >> lo); ai.lo_bits = lo; ai.n_claims = (int)d.z.size();
            ai.blk_start = acc_blk;
            acc_blk += (int)((out_len + HG_BLOCK * HG_EQACC_PER_THREAD - 1) / (HG_BLOCK * HG_EQACC_PER_THREAD));
            accs.push_back(ai);
            const int lp = eq_lo_bits(d.pt.size());
            auto point = [&](const std::vector<X>& p) {
                const size_t off = flat.size();
                flat.insert(flat.end(), p.begin(), p.end());
                return split(off, (int)p.size(), lp, std::string::npos, 0);
            };
            const EqSplitItem<FP> sp = point(d.pt);
            Ref r = {w_pool_.p + woff, sp.eq_lo, sp.eq_hi, nullptr, nullptr, lp};
            if (d.kind == DC_GENERAL) {  // u and v: both phases run over the same S entries
                const EqSplitItem<FP> sv = point(d.v);
                r.vlo = sv.eq_lo; r.vhi = sv.eq_hi;
            }
            refs.push_back(r);
            woff += out_len;
        }
        d_pts = sc_.stage(flat);
        for (size_t i = 0; i < splits.size(); i++) {
            splits[i].point = d_pts + offs[i].first;
            if (offs[i].second != std::string::npos) splits[i].alpha = d_pts + offs[i].second;
        }
        HG_K(ctx_, KC_GKR_PREP, eoff * sizeof(X), k_eq_split_multi<FP><<<split_blk, HG_BLOCK, 0, s>>>(sc_.stage(splits), (int)splits.size()));
        HG_K(ctx_, KC_GKR_PREP, woff * sizeof(X), k_eq_accumulate<FP><<<acc_blk, HG_BLOCK, 0, s>>>(sc_.stage(accs), (int)accs.size()));
        // FFT weights: transform(W) in place, batched by (size, direction)
        std::map<std::pair<int, int>, std::vector<X*>> ffts;
        for (size_t g = 0; g < group.size(); g++) {
            const DeferredCheck<FP>& d = *qs[group[g]];
            if (d.kind == DC_FFT) ffts[{(int)d.z[0].size(), desc_.node_fft_inverse(d.index) ? 1 : 0}].push_back(refs[g].w);
        }
        for (auto& kv : ffts) {
            const int lg = kv.first.first;
            const size_t N = (size_t)1 << lg, cnt = kv.second.size();
            if (planes_.n < FP::PLANES * N * cnt) { HG_CUDA(cudaStreamSynchronize(s)); planes_.alloc(FP::PLANES * N * cnt); }
            X* const* d_tabs = sc_.stage(kv.second);
            HG_K(ctx_, KC_GKR_PREP, N * cnt * sizeof(X) * 2, k_ext_split<FP><<<dim3((unsigned)((N + 255) / 256), (unsigned)cnt), 256, 0, s>>>(d_tabs, N, planes_.p));
            ntt_->run(planes_.p, lg, kv.first.second != 0, FP::PLANES * cnt);
            HG_K(ctx_, KC_GKR_PREP, N * cnt * sizeof(X) * 2, k_ext_merge<FP><<<dim3((unsigned)((N + 255) / 256), (unsigned)cnt), 256, 0, s>>>(planes_.p, N, d_tabs));
        }
        std::vector<DotItem<FP, X>> dots;
        std::vector<EdgeItem<FP>> edges;
        std::vector<MulEdgeItem<FP>> muls;
        int dot_blk = 0, edge_blk = 0, mul_blk = 0;
        size_t dot_bytes = 0, edge_bytes = 0, mul_bytes = 0, pblk = 0;
        auto edge_blocks = [&](size_t n) { return (int)std::max<size_t>(1, std::min<size_t>((n + HG_BLOCK * 8 - 1) / (HG_BLOCK * 8), 2 * (size_t)ctx_->sm_count)); };
        for (size_t g = 0; g < group.size(); g++) {
            const DeferredCheck<FP>& d = *qs[group[g]];
            const Ref& r = refs[g];
            if (d.kind == DC_FFT) {
                DotItem<FP, X> it;
                it.t = r.w; it.eq_lo = r.plo; it.eq_hi = r.phi; it.out = sc_.out.p + 3 * g; it.partials = sc_.partials.p + 2 * pblk; it.counter = sc_.counters.p + g;
                it.n = desc_.node_out_len(d.index); it.lo_bits = r.lp; it.blk_start = dot_blk;
                it.nblk = (int)std::min<size_t>(it.n >> r.lp, (size_t)ctx_->sm_count);
                dot_blk += it.nblk; pblk += it.nblk; dot_bytes += it.n * sizeof(X);
                dots.push_back(it);
                continue;
            }
            const Edges& E = edges_.at(d.index);
            EdgeItem<FP> it;
            it.out_idx = E.out_idx.p; it.in_idx = E.in_idx.p; it.coef = E.coef.p; it.w = r.w; it.eq_lo = r.plo; it.eq_hi = r.phi;
            it.out = sc_.out.p + 3 * g; it.partials = sc_.partials.p + 2 * pblk; it.counter = sc_.counters.p + g;
            it.n = E.n; it.lo_bits = r.lp; it.blk_start = edge_blk; it.nblk = edge_blocks(E.n);
            edge_blk += it.nblk; pblk += it.nblk; edge_bytes += E.n * (2 * sizeof(u32) + sizeof(B) + sizeof(X));
            edges.push_back(it);
            if (d.kind != DC_GENERAL) continue;
            // counter g again: k_edge_sum has returned it to 0 before k_mul_edge_sum starts on the same stream
            const MulEdges& M = mul_edges_.at(d.index);
            MulEdgeItem<FP> mt;
            mt.out_idx = M.out_idx.p; mt.x_idx = M.x_idx.p; mt.y_idx = M.y_idx.p; mt.coef = M.coef.p; mt.w = r.w;
            mt.equ_lo = r.plo; mt.equ_hi = r.phi; mt.eqv_lo = r.vlo; mt.eqv_hi = r.vhi;
            mt.out = sc_.out.p + 3 * g + 2; mt.partials = sc_.partials.p + 2 * pblk; mt.counter = sc_.counters.p + g;
            mt.n = M.n; mt.lo_bits = r.lp; mt.blk_start = mul_blk; mt.nblk = edge_blocks(M.n);
            mul_blk += mt.nblk; pblk += mt.nblk; mul_bytes += M.n * (3 * sizeof(u32) + sizeof(B) + sizeof(X));
            muls.push_back(mt);
        }
        if (!dots.empty()) HG_K(ctx_, KC_DOT, dot_bytes, k_dot_eq_items<FP, X><<<dot_blk, HG_BLOCK, 0, s>>>(sc_.stage(dots), (int)dots.size()));
        if (!edges.empty()) HG_K(ctx_, KC_GKR_PREP, edge_bytes, k_edge_sum<FP><<<edge_blk, HG_BLOCK, 0, s>>>(sc_.stage(edges), (int)edges.size()));
        if (!muls.empty()) HG_K(ctx_, KC_GKR_PREP, mul_bytes, k_mul_edge_sum<FP><<<mul_blk, HG_BLOCK, 0, s>>>(sc_.stage(muls), (int)muls.size()));
        sc_.finish(3 * group.size());
        for (size_t g = 0; g < group.size(); g++) {
            const int kind = qs[group[g]]->kind, slots = kind == DC_FFT ? 1 : kind == DC_LINEAR ? 2 : 3;
            for (int j = 0; j < slots; j++) q[group[g]][j] = sc_.h_out.p[3 * g + j];
        }
    }

    DeviceCtx* ctx_;
    NttEngine<FP>* ntt_;
    GkrVerifierHost<FP> desc_;
    size_t max_batch_;
    VerifyScratch<FP> sc_;
    std::vector<size_t> input_lens_;
    std::map<int, Edges> edges_;          // linear and general layers
    std::map<int, MulEdges> mul_edges_;   // general layers
    DevBuf<B> subtables_;
    size_t subtable_len_ = 0;
    double timing_us_[3] = {0, 0, 0};
    DevBuf<X> w_pool_;
    DevBuf<B> planes_;
};

}  // namespace hg
