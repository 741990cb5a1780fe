// Device GKR prover for the circuits bfv-gkr builds: Circuit::{insert, connect, evaluate} and gkr::prove_gkr
// (call sites /root/reference/bfv-gkr/src/sk_encryption_circuit.rs:102-290, :442, :455-457). The engine is the un-vendored `gkr`
// crate (PARITY UNPINNED); the protocol restated here is specified in DESIGN.md section 3 (the parity tests check it against an independent CPU restatement):
//     per node, in reverse topological order: [T > 1 claims: squeeze alpha] -> product sumcheck rounds -> write input evaluations
// Node shapes: Input, Vanilla with linear gates (relay / scale / add-const / sum), the element-wise product layer, general
// Vanilla layers (any other product terms: two sumchecks, DESIGN.md section 7b, A11), FFT forward / inverse, Lasso. In
// PREFETCH mode every node's sumcheck is independent (claim POINTS are transcript challenges, only claim VALUES flow between
// nodes, and those are needed on the host only), so round j of all nodes is one launch.
#pragma once
#include <algorithm>
#include <map>

#include "gkr_kernels.cuh"
#include "ntt_engine.cuh"

namespace hg {

enum GkrNodeKind { GKR_INPUT = 0, GKR_VANILLA = 1, GKR_FFT = 2, GKR_LASSO = 3 };

// host description of one Vanilla layer (VanillaNode::new(input_arity, log2_sub_input_size, gates, num_reps)), CSR over gates
struct VanillaDesc {
    size_t arity = 0, log2_sub = 0, num_reps = 1, n_gates = 0;
    std::vector<uint8_t> has_const;
    std::vector<uint64_t> consts;                       // limbs per gate
    std::vector<uint64_t> add_ptr, add_coef, add_wire;  // add_coef: limbs
    std::vector<uint32_t> add_in;
    std::vector<uint64_t> mul_ptr, mul_coef, mul_w0, mul_w1;
    std::vector<uint32_t> mul_in0, mul_in1;
};

template <class FP> class GkrCircuitDev {
  public:
    typedef typename FP::B B;
    typedef typename FP::X X;

    struct InputClaim { std::vector<X> point; X value; };

    GkrCircuitDev(DeviceCtx* ctx, NttEngine<FP>* ntt) : ctx_(ctx), ntt_(ntt) {}

    int insert_input(size_t log2_size, size_t num_reps) {
        auto n = std::make_unique<Node>();
        n->kind = GKR_INPUT; n->out_len = num_reps << log2_size;
        nodes_.push_back(std::move(n));
        return (int)nodes_.size() - 1;
    }
    int insert_fft(size_t log2_size, bool inverse) {
        auto n = std::make_unique<Node>();
        n->kind = GKR_FFT; n->out_len = (size_t)1 << log2_size; n->fft_inverse = inverse; n->log2_size = (int)log2_size;
        n->value.alloc(n->out_len);
        nodes_.push_back(std::move(n));
        return (int)nodes_.size() - 1;
    }
    int insert_lasso(LassoNodeDev<FP>* lasso) {
        auto n = std::make_unique<Node>();
        n->kind = GKR_LASSO; n->out_len = 1; n->lasso = lasso;
        nodes_.push_back(std::move(n));
        return (int)nodes_.size() - 1;
    }
    int insert_vanilla(const VanillaDesc& d) {
        auto np = std::make_unique<Node>();
        Node& n = *np;
        n.kind = GKR_VANILLA; n.arity = (int)d.arity; n.log2_sub = (int)d.log2_sub; n.num_reps = (int)d.num_reps; n.ng = d.n_gates;
        n.out_len = pad2(d.n_gates * d.num_reps);
        n.n_in = d.num_reps << d.log2_sub;
        n.a_pad = pad2(d.arity);
        const size_t ng = d.n_gates, sub = (size_t)1 << d.log2_sub;
        // the CSR comes from the caller: validate it before it indexes host arrays here and device arrays in the kernels
        if (d.arity < 1 || d.arity > 4096 || d.log2_sub > 40 || d.num_reps < 1 || ng < 1) throw std::runtime_error("VanillaNode: bad shape");
        if (d.add_ptr.size() != ng + 1 || d.mul_ptr.size() != ng + 1 || d.has_const.size() != ng) throw std::runtime_error("VanillaNode: CSR pointer arrays must have n_gates + 1 entries");
        if (d.add_ptr[0] != 0 || d.mul_ptr[0] != 0) throw std::runtime_error("VanillaNode: CSR pointers must start at 0");
        for (size_t g = 0; g < ng; g++)
            if (d.add_ptr[g + 1] < d.add_ptr[g] || d.mul_ptr[g + 1] < d.mul_ptr[g]) throw std::runtime_error("VanillaNode: CSR pointers must be non-decreasing");
        const size_t n_add = d.add_ptr[ng], n_mul = d.mul_ptr[ng];
        if (d.add_in.size() < n_add || d.add_wire.size() < n_add || d.add_coef.size() < n_add * FP::B_LIMBS) throw std::runtime_error("VanillaNode: additive edge arrays are shorter than add_ptr[n_gates]");
        if (d.mul_in0.size() < n_mul || d.mul_in1.size() < n_mul || d.mul_w0.size() < n_mul || d.mul_w1.size() < n_mul || d.mul_coef.size() < n_mul * FP::B_LIMBS)
            throw std::runtime_error("VanillaNode: multiplicative edge arrays are shorter than mul_ptr[n_gates]");
        for (size_t e = 0; e < n_add; e++)
            if (d.add_in[e] >= d.arity || d.add_wire[e] >= sub) throw std::runtime_error("VanillaNode: additive edge " + std::to_string(e) + " points outside the inputs");
        for (size_t e = 0; e < n_mul; e++)
            if (d.mul_in0[e] >= d.arity || d.mul_in1[e] >= d.arity || d.mul_w0[e] >= sub || d.mul_w1[e] >= sub)
                throw std::runtime_error("VanillaNode: multiplicative edge " + std::to_string(e) + " points outside the inputs");
        // classify
        n.is_linear = n_mul == 0;
        n.is_elemmul = false;
        if (!n.is_linear) {
            bool ok = d.arity == 2 && n_add == 0 && n_mul == ng && d.num_reps == 1;
            for (size_t g = 0; ok && g < ng; g++) {
                ok = !d.has_const[g] && d.mul_ptr[g] == g && d.mul_in0[g] == 0 && d.mul_in1[g] == 1 && d.mul_w0[g] == g && d.mul_w1[g] == g &&
                     FP::b_eq(FP::b_from_limbs(&d.mul_coef[g * FP::B_LIMBS]), FP::b_one());
            }
            n.is_elemmul = ok;
            n.is_general = !ok;  // any other product term: the two-phase layer sumcheck (DESIGN.md section 3, A11)
        }
        auto up = [](auto& buf, const auto& v) { buf.alloc(std::max<size_t>(v.size(), 1)); if (!v.empty()) HG_CUDA(cudaMemcpy(buf.p, v.data(), v.size() * sizeof(v[0]), cudaMemcpyHostToDevice)); };
        std::vector<B> addc(n_add), mulc(n_mul), cg(ng);
        for (size_t e = 0; e < n_add; e++) addc[e] = FP::b_from_limbs(&d.add_coef[e * FP::B_LIMBS]);
        for (size_t e = 0; e < n_mul; e++) mulc[e] = FP::b_from_limbs(&d.mul_coef[e * FP::B_LIMBS]);
        n.has_consts = false;
        for (size_t g = 0; g < ng; g++) { cg[g] = d.has_const[g] ? FP::b_from_limbs(&d.consts[g * FP::B_LIMBS]) : FP::b_zero(); if (d.has_const[g]) n.has_consts = true; }
        up(n.add_ptr, d.add_ptr); up(n.add_in, d.add_in); up(n.add_wire, d.add_wire); up(n.add_coef, addc);
        up(n.mul_ptr, d.mul_ptr); up(n.mul_in0, d.mul_in0); up(n.mul_w0, d.mul_w0); up(n.mul_in1, d.mul_in1); up(n.mul_w1, d.mul_w1); up(n.mul_coef, mulc);
        up(n.consts, cg);
        {   // forward runs (k_vanilla_runs): maximal stretches of gates with the same number of edge slots, every slot walking one input
            // wire by wire with one coefficient, and the same constant
            typedef typename Node::FwdRun FwdRun;
            bool ok = true;
            if (n.is_elemmul) {
                FwdRun r; r.g0 = 0; r.len = ng; r.ne = -2; r.cst = FP::b_zero();
                r.in[0] = 0; r.in[1] = 1; r.w0[0] = r.w0[1] = 0; r.coef[0] = r.coef[1] = FP::b_one();
                n.fwd_runs.push_back(r);
            } else if (n.is_linear) {
                for (size_t g = 0; ok && g < ng; g++) {
                    const uint64_t e0 = d.add_ptr[g], ne = d.add_ptr[g + 1] - e0;
                    if (ne > (uint64_t)HG_FWD_MAXE) { ok = false; break; }
                    FwdRun* last = n.fwd_runs.empty() ? nullptr : &n.fwd_runs.back();
                    bool ext = last && (uint64_t)last->ne == ne && FP::b_eq(last->cst, cg[g]);
                    for (uint64_t e = 0; ext && e < ne; e++)
                        ext = last->in[e] == d.add_in[e0 + e] && last->w0[e] + (g - last->g0) == d.add_wire[e0 + e] && FP::b_eq(last->coef[e], addc[e0 + e]);
                    if (ext) { last->len++; continue; }
                    FwdRun r; r.g0 = g; r.len = 1; r.ne = (int)ne; r.cst = cg[g];
                    for (uint64_t e = 0; e < ne; e++) { r.in[e] = d.add_in[e0 + e]; r.w0[e] = d.add_wire[e0 + e]; r.coef[e] = addc[e0 + e]; }
                    n.fwd_runs.push_back(r);
                    if (n.fwd_runs.size() * d.num_reps > 4096) ok = false;
                }
            }
            if (!ok) n.fwd_runs.clear();
        }
        if (!n.is_elemmul) {
            // reverse wiring: for every element x of the concatenated inputs, the (output, coefficient) pairs that read it
            const size_t S = n.a_pad * n.n_in;
            std::vector<uint64_t> rp(S + 1, 0);
            for (size_t r = 0; r < d.num_reps; r++)
                for (size_t g = 0; g < ng; g++)
                    for (uint64_t e = d.add_ptr[g]; e < d.add_ptr[g + 1]; e++) rp[(size_t)d.add_in[e] * n.n_in + r * sub + d.add_wire[e] + 1]++;
            for (size_t x = 0; x < S; x++) rp[x + 1] += rp[x];
            std::vector<uint32_t> ro(rp[S]);
            std::vector<B> rc(rp[S]);
            std::vector<uint64_t> fill(rp.begin(), rp.end() - 1);
            for (size_t r = 0; r < d.num_reps; r++)
                for (size_t g = 0; g < ng; g++)
                    for (uint64_t e = d.add_ptr[g]; e < d.add_ptr[g + 1]; e++) {
                        size_t x = (size_t)d.add_in[e] * n.n_in + r * sub + d.add_wire[e];
                        ro[fill[x]] = (uint32_t)(r * ng + g); rc[fill[x]] = addc[e]; fill[x]++;
                    }
            up(n.rev_ptr, rp); up(n.rev_out, ro); up(n.rev_coef, rc);
            // piecewise-identity wiring (k_wiring_runs): maximal runs of elements with one reader each, consecutive outputs, one coefficient
            bool compressible = true;
            typedef typename Node::WireRun WireRun;
            for (size_t x = 0; compressible && x < S; x++) {
                const uint64_t deg = rp[x + 1] - rp[x];
                if (deg > 1) { compressible = false; break; }
                WireRun* last = n.wire_runs.empty() ? nullptr : &n.wire_runs.back();
                if (deg == 0) {
                    if (last && last->kind == 0) last->len++;
                    else n.wire_runs.push_back(WireRun{x, 1, 0, 0, FP::b_zero()});
                } else {
                    const uint32_t o = ro[rp[x]];
                    const B c = rc[rp[x]];
                    if (last && last->kind != 0 && (uint64_t)last->out0 + last->len == o && FP::b_eq(last->coef, c)) last->len++;
                    else n.wire_runs.push_back(WireRun{x, 1, o, FP::b_eq(c, FP::b_one()) ? 1 : 2, c});
                }
                if (n.wire_runs.size() > 4096) compressible = false;  // not worth a descriptor per run
            }
            if (!compressible) n.wire_runs.clear();
            if (n.has_consts) {
                std::vector<B> cf(n.out_len, FP::b_zero());
                for (size_t r = 0; r < d.num_reps; r++) for (size_t g = 0; g < ng; g++) cf[r * ng + g] = cg[g];
                up(n.consts_full, cf);
            }
        }
        if (n.is_general) {
            // the product terms keyed by either side: row x of the x-keyed CSR = (y, output, coefficient) of every term that reads x as
            // its first factor, row y of the y-keyed CSR = (x, output, coefficient); indices are positions in the concatenated inputs
            const size_t S = n.a_pad * n.n_in;
            if (S > ((size_t)1 << 32) || n.out_len > ((size_t)1 << 32) || n_mul * d.num_reps > ((size_t)1 << 32)) throw std::runtime_error("VanillaNode: general layer too large");
            auto pos = [&](uint32_t in, size_t r, uint64_t w) { return (size_t)in * n.n_in + r * sub + w; };
            std::vector<uint64_t> px(S + 1, 0), py(S + 1, 0);
            for (size_t r = 0; r < d.num_reps; r++)
                for (size_t e = 0; e < n_mul; e++) { px[pos(d.mul_in0[e], r, d.mul_w0[e]) + 1]++; py[pos(d.mul_in1[e], r, d.mul_w1[e]) + 1]++; }
            for (size_t x = 0; x < S; x++) { px[x + 1] += px[x]; py[x + 1] += py[x]; }
            const size_t ne = px[S];
            std::vector<uint32_t> xo(ne), xout(ne), yo(ne), yout(ne);
            std::vector<B> xc(ne), yc(ne);
            std::vector<uint64_t> fx(px.begin(), px.end() - 1), fy(py.begin(), py.end() - 1);
            for (size_t r = 0; r < d.num_reps; r++)
                for (size_t g = 0; g < ng; g++)
                    for (uint64_t e = d.mul_ptr[g]; e < d.mul_ptr[g + 1]; e++) {
                        const size_t x = pos(d.mul_in0[e], r, d.mul_w0[e]), y = pos(d.mul_in1[e], r, d.mul_w1[e]);
                        const uint32_t o = (uint32_t)(r * ng + g);
                        xo[fx[x]] = (uint32_t)y; xout[fx[x]] = o; xc[fx[x]] = mulc[e]; fx[x]++;
                        yo[fy[y]] = (uint32_t)x; yout[fy[y]] = o; yc[fy[y]] = mulc[e]; fy[y]++;
                    }
            up(n.gx_ptr, px); up(n.gx_other, xo); up(n.gx_out, xout); up(n.gx_coef, xc);
            up(n.gy_ptr, py); up(n.gy_other, yo); up(n.gy_out, yout); up(n.gy_coef, yc);
            n.n_terms = ne;
        }
        n.value.alloc(n.out_len);
        HG_CUDA(cudaDeviceSynchronize());  // blocking uploads from pageable memory vs non-blocking streams (see LassoNodeDev's constructor)
        nodes_.push_back(std::move(np));
        return (int)nodes_.size() - 1;
    }
    void connect(int from, int to) {
        if (from < 0 || to < 0 || from >= (int)nodes_.size() || to >= (int)nodes_.size()) throw std::runtime_error("connect: no such node");
        nodes_[to]->preds.push_back(from);
        nodes_[from]->succs.push_back(to);
        topo_.clear();
        eval_planned_ = false;
    }
    size_t num_nodes() const { return nodes_.size(); }
    std::vector<size_t> input_lens() const {  // output length of every input node, insertion order
        std::vector<size_t> v;
        for (auto& n : nodes_) if (n->kind == GKR_INPUT) v.push_back(n->out_len);
        return v;
    }
    // host phases of the last prove, microseconds: [witness enqueue, squeeze + upload challenges, protocol walk (+ Lasso enqueue),
    // batched layer enqueue, wait for the GPU, serialise]
    const double* timing() const { return timing_; }
    size_t total_challenges() const { return total_chal_; }
    size_t node_out_len(int id) const { return nodes_.at(id)->out_len; }
    const B* node_value(int id) const { return nodes_.at(id)->value_ptr; }

    // Circuit::evaluate (sk_encryption_circuit.rs:442): inputs = device pointers for the input nodes in insertion order.
    // Nodes are processed level by level (level = longest path from an input); the FFT nodes of one level with the same size
    // and direction share one contiguous arena and are transformed by ONE batched NTT (the circuit has 2K+1 forward
    // transforms on one level). Nothing here waits for the device.
    void evaluate(const std::vector<const B*>& inputs) {
        NvtxSpan span("eval circuit");  // sk_encryption_circuit.rs:442
        cudaStream_t s = ctx_->stream;
        size_t next = 0;
        for (auto& n : nodes_) if (n->kind == GKR_INPUT) { if (next >= inputs.size()) throw std::runtime_error("evaluate: too few inputs"); n->value_ptr = inputs[next++]; }
        if (next != inputs.size()) throw std::runtime_error("evaluate: too many inputs");
        plan_evaluate();
        for (auto& lvl : eval_levels_) {
            for (auto& grp : lvl.fft_groups) {
                const Node& first = *nodes_[grp.nodes[0]];
                const size_t N = first.out_len;
                for (size_t k = 0; k < grp.nodes.size(); k++) {
                    Node& n = *nodes_[grp.nodes[k]];
                    const Node& p = *nodes_[n.preds.at(0)];
                    HG_CUDA(cudaMemcpyAsync(grp.arena->p + k * N, p.value_ptr, N * sizeof(B), cudaMemcpyDeviceToDevice, s));
                    n.value_ptr = grp.arena->p + k * N;
                }
                ntt_->run(grp.arena->p, first.log2_size, first.fft_inverse, grp.nodes.size());
            }
            std::vector<FwdRunItem<FP>> fitems;  // every layer of this level whose gates come in runs: one launch
            int fblk = 0;
            size_t fbytes = 0;
            for (int id : lvl.vanilla) {
                Node& n = *nodes_[id];
                if (n.fwd_runs.empty()) continue;
                const size_t sub = (size_t)1 << n.log2_sub;
                auto push = [&](FwdRunItem<FP>& it) {
                    it.blk_start = fblk;
                    fblk += (int)((it.n + (size_t)HG_BLOCK * HG_FWD_PER_THREAD - 1) / ((size_t)HG_BLOCK * HG_FWD_PER_THREAD));
                    fitems.push_back(it);
                };
                for (int r = 0; r < n.num_reps; r++)
                    for (const typename Node::FwdRun& fr : n.fwd_runs) {
                        FwdRunItem<FP> it;
                        it.out = n.value.p + (size_t)r * n.ng + fr.g0; it.n = fr.len; it.ne = fr.ne; it.cst = fr.cst;
                        for (int e = 0; e < HG_FWD_MAXE; e++) { it.in[e] = nullptr; it.coef[e] = FP::b_zero(); }
                        for (int e = 0; e < (fr.ne == -2 ? 2 : fr.ne); e++) { it.in[e] = nodes_[n.preds.at(fr.in[e])]->value_ptr + (size_t)r * sub + fr.w0[e]; it.coef[e] = fr.coef[e]; }
                        push(it);
                    }
                if (n.out_len > n.ng * (size_t)n.num_reps) {  // padding up to the power of two
                    FwdRunItem<FP> it;
                    it.out = n.value.p + n.ng * (size_t)n.num_reps; it.n = n.out_len - n.ng * (size_t)n.num_reps; it.ne = 0; it.cst = FP::b_zero();
                    for (int e = 0; e < HG_FWD_MAXE; e++) { it.in[e] = nullptr; it.coef[e] = FP::b_zero(); }
                    push(it);
                }
                fbytes += n.out_len * sizeof(B) * 2;
                n.value_ptr = n.value.p;
            }
            if (!fitems.empty()) {
                // own staging buffers (the prover resets its descriptor ring per proof); re-uploaded only when a pointer changed
                const size_t bytes = fitems.size() * sizeof(FwdRunItem<FP>);
                if (!lvl.h_items) { lvl.h_items.reset(new PinnedBuf<unsigned char>()); lvl.d_items.reset(new DevBuf<unsigned char>()); }
                if (lvl.h_items->n < bytes) { HG_CUDA(cudaStreamSynchronize(s)); lvl.h_items->alloc(bytes); lvl.d_items->alloc(bytes); lvl.items_bytes = 0; }
                if (lvl.items_bytes != bytes || memcmp(lvl.h_items->p, fitems.data(), bytes) != 0) {
                    if (lvl.items_bytes) HG_CUDA(cudaStreamSynchronize(s));  // an earlier upload from this buffer may still be pending
                    memcpy(lvl.h_items->p, fitems.data(), bytes);
                    HG_CUDA(cudaMemcpyAsync(lvl.d_items->p, lvl.h_items->p, bytes, cudaMemcpyHostToDevice, s));
                    lvl.items_bytes = bytes;
                }
                HG_K(ctx_, KC_MISC, fbytes, k_vanilla_runs<FP><<<fblk, HG_BLOCK, 0, s>>>((const FwdRunItem<FP>*)lvl.d_items->p, (int)fitems.size()));
            }
            for (int id : lvl.vanilla) {
                Node& n = *nodes_[id];
                if (!n.fwd_runs.empty()) continue;
                bool changed = false;
                for (size_t k = 0; k < n.preds.size(); k++) {
                    const B* p = nodes_[n.preds[k]]->value_ptr;
                    if (n.h_in_ptrs.p[k] != p) { n.h_in_ptrs.p[k] = p; changed = true; }
                }
                if (changed) HG_CUDA(cudaMemcpyAsync(n.in_ptrs.p, n.h_in_ptrs.p, n.preds.size() * sizeof(B*), cudaMemcpyHostToDevice, s));
                VanillaFwd w{n.add_ptr.p, n.add_in.p, n.add_wire.p, n.mul_ptr.p, n.mul_in0.p, n.mul_w0.p, n.mul_in1.p, n.mul_w1.p};
                HG_K(ctx_, KC_MISC, n.out_len * sizeof(B) * 2,
                     k_vanilla_eval<FP><<<(unsigned)((n.out_len + 255) / 256), 256, 0, s>>>(w, n.add_coef.p, n.mul_coef.p, n.consts.p, (const B* const*)n.in_ptrs.p, n.ng,
                                                                                          (size_t)1 << n.log2_sub, n.num_reps, n.out_len, n.value.p));
                n.value_ptr = n.value.p;
            }
        }
        evaluated_ = true;
    }

    // gkr::prove_gkr (sk_encryption_circuit.rs:455-457). output_claims: one per output node (nodes without successors, insertion
    // order), point given by value (the caller squeezed it from the same transcript). Returns the claims on the input nodes.
    std::vector<std::vector<InputClaim>> prove(Keccak256Transcript<FP>& tr, ProveMode mode, const WireOptions& wo,
                                               const std::vector<InputClaim>& output_claims) {
        if (!tr.prefetch_legal()) mode = kModeInteractive;
        enqueue(tr, mode, wo, output_claims, 0, 1);
        ch_->flush(&timing_[4], &timing_[5]);
        return collect();
    }
    // ---- ONE gkr::prove_gkr over `world` devices (SURVEY.md 8e). With prefetched challenges every node's claim reduction is
    // an independent job whose messages land in disjoint slots of one message buffer, except the Lasso node's grand-product
    // round polynomials, which are sums over its 2m vectors. Device `rank` runs the generic node sumchecks q with q % world ==
    // rank and its share of the Lasso node (LassoNodeDev::set_shard), leaves every other slot zero, and copies its buffer into
    // d_out; the element-wise field sum over devices (one all-gather of shard_message_count() elements + k_shard_merge) is the
    // buffer a single device produces, which rank 0 serialises with emit_shard_dev. Nothing here waits for the device.
    size_t prove_shard_dev(Keccak256Transcript<FP>& tr, const WireOptions& wo, const std::vector<InputClaim>& output_claims, int rank, int world, X* d_out,
                           size_t cap) {
        if (world < 1 || rank < 0 || rank >= world) throw std::runtime_error("prove_gkr: bad shard rank / world size");
        if (!tr.prefetch_legal()) throw std::runtime_error("prove_gkr: a sharded proof needs a transcript whose challenges do not depend on the messages");
        enqueue(tr, kModePrefetch, wo, output_claims, rank, world);
        return ch_->copy_partial_to(d_out, cap);
    }
    std::vector<std::vector<InputClaim>> emit_shard_dev(const X* d_merged, size_t count) {
        ch_->emit_merged(d_merged, count);
        return collect();
    }
    // the same with the serialisation split over the devices: device `part` returns the bytes of its range of the proof (the caller
    // concatenates the ranges in order and appends them to rank 0's transcript); the input claims are valid on every device
    std::vector<std::vector<InputClaim>> emit_shard_part_dev(const X* d_merged, size_t count, int part, int nparts, std::vector<uint8_t>& bytes) {
        ch_->emit_merged_device_part(d_merged, count, part, nparts, bytes);
        return collect();
    }
    size_t shard_message_count() { plan(); return msg_budget_; }

  private:
    struct Claim { bool by_index; size_t idx; std::vector<X> point_host; int nvars; std::shared_ptr<X> value; };
    std::vector<std::vector<Claim>> pending_claims_;
    size_t msg_budget_ = 0;
    // the claims that reached the input nodes (what verify() checks, sk_encryption_circuit.rs:512-516), after the messages are on the host
    std::vector<std::vector<InputClaim>> collect() {
        Channel<FP>& ch = *ch_;
        if (ch.chal_used() != total_chal_) throw std::runtime_error("prove_gkr: challenge count mismatch");
        std::vector<std::vector<InputClaim>> res;
        for (size_t i = 0; i < nodes_.size(); i++) {
            if (nodes_[i]->kind != GKR_INPUT) continue;
            std::vector<InputClaim> v;
            for (auto& c : pending_claims_[i]) {
                InputClaim ic;
                if (c.by_index) { ic.point.resize(c.nvars); for (int q = 0; q < c.nvars; q++) ic.point[q] = ch.chal(c.idx + q); }
                else ic.point = c.point_host;
                ic.value = *c.value;
                v.push_back(ic);
            }
            res.push_back(v);
        }
        return res;
    }
    // everything of prove() up to (not including) the download of the messages
    void enqueue(Keccak256Transcript<FP>& tr, ProveMode mode, const WireOptions& wo, const std::vector<InputClaim>& output_claims, int rank, int world) {
        if (!evaluated_) throw std::runtime_error("prove_gkr: evaluate the circuit first");
        NvtxSpan span("GKR prove");     // sk_encryption_circuit.rs:455
        const bool sharded = world > 1;
        cudaStream_t s = ctx_->stream;
        auto now = []() { return std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
        const double t0 = now();
        plan();
        desc_off_ = 0; eq_off_ = 0;  // the previous proof ended with a synchronised flush: its staging regions are free
        Channel<FP>& ch = *ch_;
        if (sharded) ch.zero_messages();  // slots this device does not own must read as zero in the sum over devices
        pending_claims_.assign(nodes_.size(), {});
        std::vector<std::vector<Claim>>& claims = pending_claims_;
        struct ShardScope {  // the Lasso nodes work for this device while this call enqueues them
            GkrCircuitDev* c;
            ShardScope(GkrCircuitDev* cc, int r, int w) : c(cc) { for (auto& n : c->nodes_) if (n->kind == GKR_LASSO) n->lasso->set_shard(r, w); }
            ~ShardScope() { for (auto& n : c->nodes_) if (n->kind == GKR_LASSO) n->lasso->set_shard(0, 1); }
        } shard_scope(this, rank, world);
        // output claims: their points live in extra device slots after the challenges
        std::vector<int> outs;
        for (size_t i = 0; i < nodes_.size(); i++) if (nodes_[i]->succs.empty() && nodes_[i]->kind != GKR_INPUT) outs.push_back((int)i);
        if (outs.size() != output_claims.size()) throw std::runtime_error("prove_gkr: one output claim per output node is required");
        {
            size_t slot = 0;
            std::vector<X> stage;
            for (size_t i = 0; i < outs.size(); i++) {
                Claim c; c.by_index = false; c.idx = slot; c.point_host = output_claims[i].point; c.nvars = (int)output_claims[i].point.size();
                c.value = std::make_shared<X>(output_claims[i].value);
                slot += c.point_host.size();
                stage.insert(stage.end(), c.point_host.begin(), c.point_host.end());
                claims[outs[i]].push_back(c);
            }
            if (slot > d_outpts_.n) d_outpts_.alloc(slot + 16);
            if (slot > h_outpts_.n) h_outpts_.alloc(slot + 16);
            if (!stage.empty()) {  // pinned staging: no host wait (the previous proof's flush has synchronised the stream)
                memcpy(h_outpts_.p, stage.data(), stage.size() * sizeof(X));
                HG_CUDA(cudaMemcpyAsync(d_outpts_.p, h_outpts_.p, stage.size() * sizeof(X), cudaMemcpyHostToDevice, s));
            }
        }
        // In prefetch mode the layer sumchecks depend on nothing the Lasso node computes: they go to the context's second
        // stream, forked here (after the challenge upload) and joined before the messages are downloaded. Per-launch
        // profiling keeps everything on one stream so that launches are timed one at a time.
        const bool fork = mode == kModePrefetch && ctx_->two_streams && !ctx_->profile && ctx_->stream2 != nullptr;
        double t1 = t0;
        if (fork) {
            ch.begin(&tr, mode, total_chal_);
            HG_CUDA(cudaEventRecord(ctx_->ev_fork, s));
            t1 = now();
        }
        // Lasso witness kernels need no challenge
        for (auto& n : nodes_) if (n->kind == GKR_LASSO) {
            const Node& p = *nodes_[n->preds.at(0)];
            n->lasso->enqueue_witness(p.value_ptr, n->lasso->num_rows(), wo);
        }
        if (!fork) {
            t1 = now();
            ch.begin(&tr, mode, total_chal_);  // Keccak squeezing overlaps the witness kernels
        }
        const double t2 = now();
        auto point_ptr = [&](const Claim& c) -> const X* { return c.by_index ? ch.d_chal(c.idx) : d_outpts_.p + c.idx; };
        std::vector<Job> jobs;
        auto ord = topo();
        Channel<FP>* chp = &ch;
        for (size_t oi = ord.size(); oi-- > 0;) {
            const int id = ord[oi];
            Node& n = *nodes_[id];
            if (n.kind == GKR_INPUT) continue;
            if (n.kind == GKR_LASSO) {
                size_t r_idx = 0, sum_off = 0;
                const bool side = !sharded && ch.begin_side();  // its serialisation overlaps the layer kernels enqueued below
                n.lasso->enqueue_protocol(ch, mode, wo, &r_idx, &sum_off);
                Claim c; c.by_index = true; c.idx = r_idx; c.nvars = n.lasso->num_vars(); c.value = std::make_shared<X>(FP::x_zero());
                auto vp = c.value;
                ch.emit([chp, vp, sum_off]() { *vp = chp->msg(sum_off); });
                if (side) ch.end_side();
                claims[n.preds.at(0)].push_back(c);
                continue;
            }
            auto& cl = claims[id];
            if (cl.empty()) throw std::runtime_error("prove_gkr: node without claims");
            Job job;
            job.node = id;
            job.nt = n.is_elemmul ? 2 : 1;
            job.S = n.kind == GKR_FFT || n.is_elemmul ? n.out_len : n.a_pad * n.n_in;
            job.nv = log2sz(job.S);
            job.alpha_idx = cl.size() > 1 ? ch.squeeze(1) : (size_t)-1;
            for (auto& c : cl) { if (((size_t)1 << c.nvars) != n.out_len) throw std::runtime_error("prove_gkr: claim point does not match the node's output size"); job.points.push_back(point_ptr(c)); }
            job.const_off = ch.alloc_msg(1);
            auto st = std::make_shared<ScHostState<FP>>();
            {
                std::vector<std::shared_ptr<X>> vals;
                for (auto& c : cl) vals.push_back(c.value);
                const size_t aidx = job.alpha_idx, coff = job.const_off;
                const bool has_c = lin(n) && n.has_consts;
                ch.emit([chp, st, vals, aidx, coff, has_c]() {
                    X a = aidx == (size_t)-1 ? FP::x_one() : chp->chal(aidx), p = FP::x_one(), comb = FP::x_zero();
                    for (auto& v : vals) { comb = FP::x_add(comb, FP::x_mul(p, *v)); p = FP::x_mul(p, a); }
                    if (has_c) comb = FP::x_sub(comb, chp->msg(coff));
                    st->claim = comb;
                });
            }
            run_job(ch, mode, wo, job, st, jobs);
            if (n.is_general) {
                // phase 2 over y: sum_y (X(u) M(u, y)) X(y) = X(u) H(u), u = phase 1's challenges. The device samples the rounds with the
                // unscaled M_u and reduces H(u) = sum_y M_u[y] X[y] into slot hu_off; X(u) = sum_k eq(u_hi, k) X_k(u_lo) comes from phase 1's
                // input evaluations. The claim thus depends on message slots and challenges only, not on phase 1's host state.
                const Job& p1 = jobs.back();
                Job j2;
                j2.node = id; j2.phase = 1; j2.nt = 1; j2.S = p1.S; j2.nv = p1.nv; j2.u_idx = p1.r0_idx;
                j2.hu_off = ch.alloc_msg(1);
                auto st2 = std::make_shared<ScHostState<FP>>();
                const size_t eo = p1.evals_off, hu = j2.hu_off, u0 = p1.r0_idx;
                const int m = log2sz(n.n_in), nvh = p1.nv - m, ar = n.arity;
                ch.emit([chp, st2, eo, hu, u0, m, nvh, ar]() {
                    X xu = FP::x_zero();
                    for (int k = 0; k < ar; k++) {
                        X e = FP::x_one();
                        for (int i = 0; i < nvh; i++) { const X r = chp->chal(u0 + m + i); e = FP::x_mul(e, ((k >> i) & 1) ? r : FP::x_sub(FP::x_one(), r)); }
                        xu = FP::x_add(xu, FP::x_mul(e, chp->msg(eo + k)));
                    }
                    st2->scaled = true; st2->scale = xu;
                    st2->claim = FP::x_mul(xu, chp->msg(hu));
                });
                run_job(ch, mode, wo, j2, st2, jobs);
            }
        }
        const double t3 = now();
        bool early = false;
        if (mode == kModePrefetch) {
            struct StreamSwap {  // every helper reads ctx->stream when it launches
                DeviceCtx* c; cudaStream_t main; bool on;
                StreamSwap(DeviceCtx* ctx, bool enable) : c(ctx), main(ctx->stream), on(enable) {
                    if (on) { c->stream = c->stream2; cudaStreamWaitEvent(c->stream2, c->ev_fork, 0); }
                }
                ~StreamSwap() {
                    if (on) { cudaEventRecord(c->ev_join, c->stream2); c->stream = main; cudaStreamWaitEvent(main, c->ev_join, 0); }
                }
            } swap(ctx_, fork);
            std::vector<Job> mine;  // the node sumchecks this device runs (all of them unless the proof is sharded)
            size_t q = 0;           // both phases of a general layer go to one device: phase 2 needs the weights and tables of phase 1
            for (const Job& j : jobs) {
                if (!sharded || (int)(q % (size_t)world) == rank) mine.push_back(j);
                if (!(j.phase == 0 && nodes_[j.node]->is_general)) q++;
            }
            prepare_jobs(ch, mine, wo);
            use_tail_ = true;
            struct TailOff { bool* f; ~TailOff() { *f = false; } } tail_off{&use_tail_};
            int maxv = 0;
            for (auto& j : mine) maxv = std::max(maxv, std::min(j.nv, stream_end(j)));
            for (int r = 0; r < maxv; r++) launch_round(ch, mine, r);
            launch_tail(ch, mine);
            launch_finals(ch, mine);
            early = fork && !sharded;
        }
        if (early) ch.arm_early(ctx_->ev_join);  // after the StreamSwap scope: ev_join marks the end of every node sumcheck
        const double t4 = now();
        timing_[0] = t1 - t0; timing_[1] = t2 - t1; timing_[2] = t3 - t2; timing_[3] = t4 - t3;
    }

    struct Work { DevBuf<X> wbuf0, wbuf1, tbuf0, tbuf1, capture; };
    struct Node {
        int kind = GKR_INPUT, log2_size = 0, num_reps = 1, arity = 0, log2_sub = 0;
        bool fft_inverse = false, is_linear = false, is_elemmul = false, is_general = false, has_consts = false;
        size_t ng = 0, out_len = 0, n_in = 0, a_pad = 1, n_terms = 0;  // n_terms: product terms of a general layer, num_reps expanded
        std::vector<int> preds, succs;
        struct FwdRun { uint64_t g0, len; int ne; uint32_t in[HG_FWD_MAXE]; uint64_t w0[HG_FWD_MAXE]; B coef[HG_FWD_MAXE]; B cst; };
        std::vector<FwdRun> fwd_runs;    // non-empty: the gates come in runs (k_vanilla_runs evaluates the layer)
        struct WireRun { uint64_t x0, len; uint32_t out0; int kind; B coef; };
        std::vector<WireRun> wire_runs;  // non-empty: the reverse wiring is piecewise the identity (k_wiring_runs)
        DevBuf<u64> add_ptr, add_wire, mul_ptr, mul_w0, mul_w1, rev_ptr;
        DevBuf<u32> add_in, mul_in0, mul_in1, rev_out;
        DevBuf<B> add_coef, mul_coef, consts, consts_full, rev_coef, value;
        DevBuf<const B*> in_ptrs;
        PinnedBuf<const B*> h_in_ptrs;  // what in_ptrs holds (uploaded again only when an input pointer changes)
        const B* value_ptr = nullptr;
        LassoNodeDev<FP>* lasso = nullptr;
        // general layers: the product terms as two reverse CSRs over the concatenated inputs, num_reps expanded. Row x of the
        // x-keyed one lists (y, output, coefficient) of every term that reads x on its first side; the y-keyed one (x, output, coefficient).
        DevBuf<u64> gx_ptr, gy_ptr;
        DevBuf<u32> gx_other, gx_out, gy_other, gy_out;
        DevBuf<B> gx_coef, gy_coef;
        // per-node work buffers of the layer sumcheck (wk[1]: phase 2 of a general layer, which runs next to phase 1)
        DevBuf<X> W, A, Mu;
        Work wk[2];
        DevBuf<B> Xcat;
    };
    // phase: 0 = the node's (first) sumcheck, 1 = phase 2 of a general layer (weights M_u, claim X(u) H(u), u = phase 1's challenges)
    struct Job {
        int node = 0, nt = 1, nv = 0, phase = 0;
        size_t S = 0, alpha_idx = (size_t)-1, const_off = 0, msg_off = 0, r0_idx = 0, evals_off = 0, u_idx = 0, hu_off = 0;
        std::vector<const X*> points;
    };
    // the rounds of one node sumcheck (launched here in interactive mode, batched by the caller in prefetch mode), its input
    // evaluations and the claims they put on the node's predecessors; appends the job to `jobs`
    void run_job(Channel<FP>& ch, ProveMode mode, const WireOptions& wo, Job& job, std::shared_ptr<ScHostState<FP>> st, std::vector<Job>& jobs) {
        Node& n = *nodes_[job.node];
        Channel<FP>* chp = &ch;
        const int n_ev = n.kind == GKR_FFT ? 1 : (n.is_elemmul ? 2 : n.arity);
        if (mode == kModeInteractive) prepare_jobs(ch, {job}, wo);
        for (int j = 0; j < job.nv; j++) {
            size_t off = ch.alloc_msg(4);
            if (j == 0) job.msg_off = off;
            if (mode == kModeInteractive) launch_round(ch, {job}, j);
            const size_t next_idx = ch.next_index();
            if (job.nt == 1) emit_round_slots<FP, 2>(ch, st, off, wo, j == 0, next_idx);
            else emit_round_slots<FP, 3>(ch, st, off, wo, j == 0, next_idx);
            size_t idx = ch.squeeze(1);
            if (j == 0) job.r0_idx = idx;
        }
        job.evals_off = ch.alloc_msg(n_ev);  // after the rounds: in interactive mode earlier slots have already been downloaded
        if (mode == kModeInteractive) launch_finals(ch, {job});
        // new claims on the predecessors: (point = the round challenges restricted to the input's variables, value = its evaluation)
        const int in_vars = lin(n) ? log2sz(n.n_in) : job.nv;
        std::vector<std::shared_ptr<X>> outv;
        for (int k = 0; k < n_ev; k++) {
            Claim c; c.by_index = true; c.idx = job.r0_idx; c.nvars = in_vars; c.value = std::make_shared<X>(FP::x_zero());
            outv.push_back(c.value);
            pending_claims_[n.preds.at(k)].push_back(c);
        }
        {
            const size_t eo = job.evals_off;
            ch.emit([chp, outv, eo]() {
                for (size_t k = 0; k < outv.size(); k++) { *outv[k] = chp->msg(eo + k); chp->transcript().write_felt_ext(*outv[k]); }
            });
        }
        jobs.push_back(job);
    }

    struct FftGroup { std::vector<int> nodes; std::unique_ptr<DevBuf<B>> arena; };
    struct EvalLevel {
        std::vector<FftGroup> fft_groups; std::vector<int> vanilla;
        std::unique_ptr<PinnedBuf<unsigned char>> h_items; std::unique_ptr<DevBuf<unsigned char>> d_items; size_t items_bytes = 0;  // k_vanilla_runs descriptors
    };
    // static schedule of evaluate(): levels, FFT batches, pointer tables
    void plan_evaluate() {
        if (eval_planned_) return;
        std::vector<int> depth(nodes_.size(), 0);
        int maxd = 0;
        for (int id : topo()) {
            Node& n = *nodes_[id];
            for (int p : n.preds) depth[id] = std::max(depth[id], depth[p] + 1);
            maxd = std::max(maxd, depth[id]);
        }
        eval_levels_.clear();
        eval_levels_.resize(maxd + 1);
        for (int id : topo()) {
            Node& n = *nodes_[id];
            if (n.kind == GKR_INPUT) continue;
            if (n.kind == GKR_LASSO) { n.value_ptr = nullptr; continue; }
            EvalLevel& lvl = eval_levels_[depth[id]];
            if (n.kind == GKR_FFT) {
                if (nodes_[n.preds.at(0)]->out_len != n.out_len) throw std::runtime_error("evaluate: FFT input size mismatch");
                FftGroup* g = nullptr;
                for (auto& cand : lvl.fft_groups) {
                    const Node& f = *nodes_[cand.nodes[0]];
                    if (f.log2_size == n.log2_size && f.fft_inverse == n.fft_inverse) { g = &cand; break; }
                }
                if (!g) { lvl.fft_groups.emplace_back(); g = &lvl.fft_groups.back(); }
                g->nodes.push_back(id);
                continue;
            }
            if ((int)n.preds.size() != n.arity) throw std::runtime_error("evaluate: Vanilla node arity does not match its connections");
            for (int pid : n.preds) if (nodes_[pid]->out_len != n.n_in) throw std::runtime_error("evaluate: Vanilla input size mismatch");
            n.in_ptrs.alloc(n.preds.size());
            n.h_in_ptrs.alloc(n.preds.size());
            for (size_t k = 0; k < n.preds.size(); k++) n.h_in_ptrs.p[k] = nullptr;
            lvl.vanilla.push_back(id);
        }
        for (auto& lvl : eval_levels_)
            for (auto& g : lvl.fft_groups) { g.arena.reset(new DevBuf<B>()); g.arena->alloc(g.nodes.size() * nodes_[g.nodes[0]]->out_len); }
        eval_planned_ = true;
    }

    static size_t pad2(size_t n) { size_t p = 1; while (p < n) p <<= 1; return p; }
    static int log2sz(size_t n) { int l = 0; while (((size_t)1 << l) < n) l++; return l; }
    static int eq_lo_bits(int nv) { return nv < 12 ? nv : 12; }

    const std::vector<int>& topo() {
        if (!topo_.empty() || nodes_.empty()) return topo_;
        std::vector<int> indeg(nodes_.size());
        std::vector<char> done(nodes_.size(), 0);
        for (size_t i = 0; i < nodes_.size(); i++) indeg[i] = (int)nodes_[i]->preds.size();
        for (size_t step = 0; step < nodes_.size(); step++) {
            int pick = -1;
            for (size_t i = 0; i < nodes_.size(); i++) if (!done[i] && indeg[i] == 0) { pick = (int)i; break; }
            if (pick < 0) throw std::runtime_error("circuit has a cycle");
            done[pick] = 1; topo_.push_back(pick);
            for (int sx : nodes_[pick]->succs) indeg[sx]--;
        }
        return topo_;
    }

    // challenge / message budget and per-node buffers (static per circuit)
    void plan() {
        if (planned_) return;
        size_t chal = 0, msg = 0, eq_elems = 0, items = 0;
        for (int id : topo()) {
            Node& n = *nodes_[id];
            if (n.kind == GKR_INPUT) continue;
            if (n.kind == GKR_LASSO) {
                if (n.preds.size() != 1) throw std::runtime_error("prove_gkr: the Lasso node takes exactly one input (lasso.rs:64)");
                if (nodes_[n.preds[0]]->out_len < n.lasso->num_rows()) throw std::runtime_error("prove_gkr: the Lasso node's input is shorter than its lookups");
                chal += n.lasso->total_challenges(); msg += n.lasso->message_budget();
                continue;
            }
            const size_t S = n.kind == GKR_FFT || n.is_elemmul ? n.out_len : n.a_pad * n.n_in;
            const int nv = log2sz(S), nt = n.is_elemmul ? 2 : 1;
            size_t n_claims = std::max<size_t>(1, n.succs.size());  // one claim per successor edge (upper bound: every successor pushes one)
            // a successor pushes one claim per input slot this node fills, a general layer two (at u_lo and at v_lo)
            size_t edges = 0;
            for (int sx : n.succs) for (int p : nodes_[sx]->preds) if (p == id) edges += nodes_[sx]->is_general ? 2 : 1;
            n_claims = std::max<size_t>(1, edges);
            const int phases = n.is_general ? 2 : 1;
            chal += (n_claims > 1 ? 1 : 0) + phases * nv;
            msg += phases * (1 + 4 * (size_t)nv + 8 + n.a_pad);
            eq_elems += n_claims * (((size_t)1 << eq_lo_bits(log2sz(n.out_len))) + (n.out_len >> eq_lo_bits(log2sz(n.out_len))) + 2);
            if (n.is_general) eq_elems += ((size_t)1 << eq_lo_bits(nv)) + (S >> eq_lo_bits(nv)) + 2;  // eq(u, .) of phase 2
            items += n_claims + 4 * phases;
            n.W.alloc(n.out_len);
            if (!(n.kind == GKR_VANILLA && n.is_elemmul)) n.A.alloc(S);
            for (int ph = 0; ph < phases; ph++) {
                Work& w = n.wk[ph];
                w.wbuf0.alloc(std::max<size_t>(S / 2, 1)); w.wbuf1.alloc(std::max<size_t>(S / 4, 1));
                w.tbuf0.alloc(std::max<size_t>(nt * (S / 2), 1)); w.tbuf1.alloc(std::max<size_t>(nt * (S / 4), 1));
                w.capture.alloc(n.a_pad + 2);
            }
            if (n.is_general) n.Mu.alloc(S);
            if (n.kind == GKR_VANILLA) n.Xcat.alloc(n.is_elemmul ? 2 * S : S);
        }
        total_chal_ = chal;
        msg_budget_ = msg + 64;
        ch_.reset(new Channel<FP>(ctx_, chal + 8, msg + 64));
        d_eq_.alloc(eq_elems + 64);
        d_partials_.alloc(((size_t)ctx_->sm_count * 16 + 8) * 8 * (items + 4));  // 8 sums per CTA when round 0 rides on round 1
        d_counters_.alloc(items + 64);
        HG_CUDA(cudaMemset(d_counters_.p, 0, d_counters_.bytes()));
        h_desc_.alloc(1 << 20);
        d_desc_.alloc(1 << 20);
        planned_ = true;
    }

    // descriptor staging: per call, a fresh region of the pinned/device descriptor buffers
    template <class T> const T* stage(const std::vector<T>& v) {
        size_t bytes = (v.size() * sizeof(T) + 15) & ~(size_t)15;
        if (desc_off_ + bytes > h_desc_.n) throw std::runtime_error("gkr: descriptor staging overflow");
        memcpy(h_desc_.p + desc_off_, v.data(), v.size() * sizeof(T));
        HG_CUDA(cudaMemcpyAsync(d_desc_.p + desc_off_, h_desc_.p + desc_off_, bytes, cudaMemcpyHostToDevice, ctx_->stream));
        const T* r = (const T*)(d_desc_.p + desc_off_);
        desc_off_ += bytes;
        return r;
    }

    // weights W, A and concatenated inputs for the given jobs
    void prepare_jobs(Channel<FP>& ch, const std::vector<Job>& jobs, const WireOptions& wo) {
        cudaStream_t s = ctx_->stream;
        if (jobs.size() > 1) { desc_off_ = 0; eq_off_ = 0; }
        if (desc_off_ > h_desc_.n / 2) { HG_CUDA(cudaStreamSynchronize(s)); desc_off_ = 0; eq_off_ = 0; }
        // eq factor tables of every (node, claim), then accumulation claim by claim (t = 0 initialises W)
        size_t max_claims = 0;
        struct EqRef { X* lo; X* hi; int lo_bits; };
        std::vector<std::vector<EqRef>> eqs(jobs.size());
        std::vector<EqSplitItem<FP>> splits;
        int split_blk = 0;
        size_t split_bytes = 0;
        for (size_t q = 0; q < jobs.size(); q++) {
            const Job& j = jobs[q];
            Node& n = *nodes_[j.node];
            if (j.phase == 1) {  // eq(u, .) over the S entries of the concatenated inputs, in two factors
                const int lo = eq_lo_bits(j.nv);
                const size_t need = ((size_t)1 << lo) + ((size_t)1 << (j.nv - lo));
                if (eq_off_ + need > d_eq_.n) throw std::runtime_error("gkr: eq table pool too small");
                X* elo = d_eq_.p + eq_off_;
                eq_off_ += need;
                EqSplitItem<FP> si; si.point = ch.d_chal(j.u_idx); si.eq_lo = elo; si.eq_hi = elo + ((size_t)1 << lo); si.nv = j.nv; si.lo_bits = lo;
                si.blk_start = split_blk; si.alpha = nullptr; si.t = 0;
                split_blk += (int)((need + HG_BLOCK - 1) / HG_BLOCK);
                split_bytes += need * sizeof(X);
                splits.push_back(si);
                eqs[q].push_back({elo, si.eq_hi, lo});
                continue;
            }
            const int nvw = log2sz(n.out_len), lo = eq_lo_bits(nvw);
            max_claims = std::max(max_claims, j.points.size());
            for (size_t t = 0; t < j.points.size(); t++) {
                const size_t need = ((size_t)1 << lo) + ((size_t)1 << (nvw - lo));
                if (eq_off_ + need > d_eq_.n) throw std::runtime_error("gkr: eq table pool too small");
                X* elo = d_eq_.p + eq_off_;
                X* ehi = elo + ((size_t)1 << lo);
                eq_off_ += need;
                EqSplitItem<FP> si; si.point = j.points[t]; si.eq_lo = elo; si.eq_hi = ehi; si.nv = nvw; si.lo_bits = lo; si.blk_start = split_blk;
                si.alpha = j.alpha_idx == (size_t)-1 ? nullptr : ch.d_chal(j.alpha_idx); si.t = (int)t;
                split_blk += (int)((need + HG_BLOCK - 1) / HG_BLOCK);
                split_bytes += need * sizeof(X);
                splits.push_back(si);
                eqs[q].push_back({elo, ehi, lo});
            }
        }
        if (!splits.empty()) HG_K(ctx_, KC_GKR_PREP, split_bytes, k_eq_split_multi<FP><<<split_blk, HG_BLOCK, 0, s>>>(stage(splits), (int)splits.size()));
        {
            std::vector<EqAccItem<FP>> items;
            int blk = 0;
            size_t bytes = 0;
            for (size_t q = 0; q < jobs.size(); q++) {
                const Job& j = jobs[q];
                if (j.points.empty()) continue;
                Node& n = *nodes_[j.node];
                EqAccItem<FP> it;
                it.eq0 = eqs[q][0].lo; it.lo_bits = eqs[q][0].lo_bits;
                it.stride = ((size_t)1 << it.lo_bits) + (n.out_len >> it.lo_bits);
                it.n_claims = (int)j.points.size();
                it.w = n.W.p; it.n = n.out_len; it.blk_start = blk;
                blk += (int)((n.out_len + HG_BLOCK * HG_EQACC_PER_THREAD - 1) / (HG_BLOCK * HG_EQACC_PER_THREAD));
                bytes += n.out_len * sizeof(X);
                items.push_back(it);
            }
            if (!items.empty()) HG_K(ctx_, KC_GKR_PREP, bytes, k_eq_accumulate<FP><<<blk, HG_BLOCK, 0, s>>>(stage(items), (int)items.size()));
        }
        (void)max_claims;
        // A per node
        std::vector<X*> fft_fwd, fft_inv;  // W tables whose transform is needed, grouped by size via a map below
        std::map<std::pair<int, int>, std::vector<int>> fft_groups;  // (log2 size, inverse) -> node ids
        std::vector<WiringItem<FP>> wires;
        std::vector<WireRunItem<FP>> runs;
        int run_blk = 0;
        size_t run_bytes = 0;
        std::vector<ConcatItem<FP>> cats;
        int wire_blk = 0, cat_blk = 0;
        size_t wire_bytes = 0, cat_bytes = 0;
        auto cat = [&](const B* src, B* dst, size_t cnt) {
            ConcatItem<FP> c; c.src = src; c.dst = dst; c.n = cnt; c.blk_start = cat_blk;
            cat_blk += (int)((cnt + HG_BLOCK * HG_CONCAT_PER_THREAD - 1) / (HG_BLOCK * HG_CONCAT_PER_THREAD));
            cat_bytes += cnt * sizeof(B) * 2;
            cats.push_back(c);
        };
        std::vector<GeneralItem<FP>> gitems, mitems;  // general layers: phase 1's G gather, phase 2's M_u gather
        int g_blk = 0, m_blk = 0;
        size_t g_bytes = 0, m_bytes = 0;
        std::vector<const Job*> hu_jobs;
        auto general_item = [&](const Node& n, bool phase2, int& blk, size_t& bytes) {
            GeneralItem<FP> gi;
            const size_t S = n.a_pad * n.n_in;
            gi.ptr = phase2 ? n.gy_ptr.p : n.gx_ptr.p; gi.other = phase2 ? n.gy_other.p : n.gx_other.p; gi.out = phase2 ? n.gy_out.p : n.gx_out.p;
            gi.coef = phase2 ? n.gy_coef.p : n.gx_coef.p; gi.w = n.W.p; gi.tab = tables(n); gi.dst = phase2 ? n.Mu.p : n.A.p;
            gi.eq_lo = gi.eq_hi = nullptr; gi.lo_bits = 0; gi.n = S; gi.blk_start = blk;
            blk += (int)((S + HG_BLOCK * HG_GENERAL_PER_THREAD - 1) / (HG_BLOCK * HG_GENERAL_PER_THREAD));
            // algorithmic bytes: the row pointers, every term (index, output, coefficient, W[output], X[y] or two eq factors), A read and G
            // written (phase 1) or M_u written (phase 2)
            bytes += (S + 1) * sizeof(u64) + n.n_terms * (2 * sizeof(u32) + sizeof(B) + sizeof(X) + (phase2 ? 2 * sizeof(X) : sizeof(B))) +
                     S * sizeof(X) * (phase2 ? 1 : 2);
            return gi;
        };
        for (size_t q = 0; q < jobs.size(); q++) {
            const Job& j = jobs[q];
            Node& n = *nodes_[j.node];
            if (j.phase == 1) {
                GeneralItem<FP> gi = general_item(n, true, m_blk, m_bytes);
                gi.eq_lo = eqs[q][0].lo; gi.eq_hi = eqs[q][0].hi; gi.lo_bits = eqs[q][0].lo_bits;
                mitems.push_back(gi);
                hu_jobs.push_back(&j);
                continue;
            }
            if (n.is_general) gitems.push_back(general_item(n, false, g_blk, g_bytes));
            if (n.kind == GKR_FFT) { fft_groups[{n.log2_size, n.fft_inverse ? 1 : 0}].push_back(j.node); continue; }
            if (n.is_elemmul) {
                // tables = [in0 | in1]
                const size_t S = n.out_len;
                for (int k = 0; k < 2; k++) cat(nodes_[n.preds.at(k)]->value_ptr, n.Xcat.p + k * S, S);
                continue;
            }
            const size_t S = n.a_pad * n.n_in;
            if (!n.wire_runs.empty()) {
                for (const typename Node::WireRun& r : n.wire_runs) {
                    WireRunItem<FP> ri; ri.w = n.W.p + r.out0; ri.A = n.A.p + r.x0; ri.n = r.len; ri.coef = r.coef; ri.kind = r.kind; ri.blk_start = run_blk;
                    run_blk += (int)((r.len + HG_BLOCK * HG_WIRERUN_PER_THREAD - 1) / (HG_BLOCK * HG_WIRERUN_PER_THREAD));
                    runs.push_back(ri);
                }
                run_bytes += S * sizeof(X) * 2;
            } else {
            WiringItem<FP> wi; wi.rev_ptr = n.rev_ptr.p; wi.rev_out = n.rev_out.p; wi.rev_coef = n.rev_coef.p; wi.w = n.W.p; wi.A = n.A.p; wi.n = S; wi.blk_start = wire_blk;
            wire_blk += (int)((S + HG_BLOCK * HG_WIRING_PER_THREAD - 1) / (HG_BLOCK * HG_WIRING_PER_THREAD));
            wire_bytes += S * sizeof(X) * 2;
            wires.push_back(wi);
            }
            if (n.a_pad != (size_t)n.arity) cat(nullptr, n.Xcat.p + (size_t)n.arity * n.n_in, (n.a_pad - n.arity) * n.n_in);
            if (n.arity > 1)  // a single input IS the concatenation: the sumcheck reads it in place (tables())
                for (int k = 0; k < n.arity; k++) cat(nodes_[n.preds.at(k)]->value_ptr, n.Xcat.p + (size_t)k * n.n_in, n.n_in);
            if (n.has_consts) {
                int blocks = (int)std::min<size_t>((n.out_len + HG_BLOCK - 1) / HG_BLOCK, (size_t)ctx_->sm_count * 2);
                HG_K(ctx_, KC_GKR_PREP, n.out_len * (sizeof(X) + sizeof(B)),
                     k_dot_wconst<FP><<<blocks, HG_BLOCK, 0, s>>>(n.W.p, n.consts_full.p, n.out_len, d_partials_.p, d_counters_.p, ch.d_msg(j.const_off)));
            }
        }
        if (!runs.empty()) HG_K(ctx_, KC_GKR_PREP, run_bytes, k_wiring_runs<FP><<<run_blk, HG_BLOCK, 0, s>>>(stage(runs), (int)runs.size()));
        if (!wires.empty()) HG_K(ctx_, KC_GKR_PREP, wire_bytes, k_wiring_gather<FP><<<wire_blk, HG_BLOCK, 0, s>>>(stage(wires), (int)wires.size()));
        if (!cats.empty()) HG_K(ctx_, KC_GKR_PREP, cat_bytes, k_concat_items<FP><<<cat_blk, HG_BLOCK, 0, s>>>(stage(cats), (int)cats.size()));
        // general layers, after W, A and the concatenated inputs: G = A + H in place of A (phase 1), M_u and H(u) (phase 2)
        if (!gitems.empty()) HG_K(ctx_, KC_GKR_PREP, g_bytes, k_general_g<FP><<<g_blk, HG_BLOCK, 0, s>>>(stage(gitems), (int)gitems.size()));
        if (!mitems.empty()) HG_K(ctx_, KC_GKR_PREP, m_bytes, k_general_mu<FP><<<m_blk, HG_BLOCK, 0, s>>>(stage(mitems), (int)mitems.size()));
        for (const Job* j : hu_jobs) {
            const Node& n = *nodes_[j->node];
            const size_t S = n.a_pad * n.n_in;
            int blocks = (int)std::min<size_t>((S + HG_BLOCK - 1) / HG_BLOCK, (size_t)ctx_->sm_count * 2);
            HG_K(ctx_, KC_GKR_PREP, S * (sizeof(X) + sizeof(B)),
                 k_dot_wconst<FP><<<blocks, HG_BLOCK, 0, s>>>(n.Mu.p, tables(n), S, d_partials_.p, d_counters_.p, ch.d_msg(j->hu_off)));
        }
        // FFT-matrix weights: A = transform(W) plane by plane, batched over all FFT nodes of the same size and direction
        for (auto& kv : fft_groups) {
            const int lg = kv.first.first;
            const bool inv = kv.first.second != 0;
            const size_t N = (size_t)1 << lg, cnt = kv.second.size();
            if (d_planes_.n < FP::PLANES * N * cnt) { HG_CUDA(cudaStreamSynchronize(s)); d_planes_.alloc(FP::PLANES * N * cnt); }
            std::vector<X*> wt, at;
            for (size_t q = 0; q < cnt; q++) { wt.push_back(nodes_[kv.second[q]]->W.p); at.push_back(nodes_[kv.second[q]]->A.p); }
            X* const* d_wt = stage(wt);
            X* const* d_at = stage(at);
            HG_K(ctx_, KC_GKR_PREP, N * cnt * sizeof(X) * 2, k_ext_split<FP><<<dim3((unsigned)((N + 255) / 256), (unsigned)cnt), 256, 0, s>>>(d_wt, N, d_planes_.p));
            ntt_->run(d_planes_.p, lg, inv, FP::PLANES * cnt);
            HG_K(ctx_, KC_GKR_PREP, N * cnt * sizeof(X) * 2, k_ext_merge<FP><<<dim3((unsigned)((N + 255) / 256), (unsigned)cnt), 256, 0, s>>>(d_planes_.p, N, d_at));
        }
        (void)wo;
    }

    const X* weights(const Job& j) const {
        const Node& n = *nodes_[j.node];
        if (j.phase == 1) return n.Mu.p;
        return n.kind == GKR_VANILLA && n.is_elemmul ? n.W.p : n.A.p;
    }
    const B* tables(const Node& n) const {
        if (n.kind == GKR_FFT || (lin(n) && n.arity == 1)) return nodes_[n.preds.at(0)]->value_ptr;
        return n.Xcat.p;
    }
    // sumchecks over the concatenated inputs (linear and general layers): the input evaluations are read off the table folded
    // over the low log2(n_in) variables
    static bool lin(const Node& n) { return n.kind == GKR_VANILLA && !n.is_elemmul; }
    Work& wk(const Job& j) { return nodes_[j.node]->wk[j.phase]; }

    // round r of every job that still has one
    void launch_round(Channel<FP>& ch, const std::vector<Job>& jobs, int r) {
        cudaStream_t s = ctx_->stream;
        std::vector<ProdItem<FP>> items;
        int blk = 0;
        size_t part_off = 0, bytes = 0;
        size_t round_pairs = 0;  // small rounds get one pair per thread (more CTAs), large ones up to 16 (fewer block-level reductions)
        // prefetch mode: round 0 of every job with a streamed round 1 is sampled by that round's launch (k_prod_round_multi FUSE0)
        auto fused0 = [&](const Job& j) { return use_tail_ && j.nv >= 2 && stream_end(j) >= 2; };
        for (const Job& j : jobs) if (r < j.nv && r < stream_end(j) && !(r == 0 && fused0(j))) round_pairs += r == 0 ? j.S / 2 : (j.S >> (r - 1)) / 4;
        bool any_fused = false;
        for (const Job& j : jobs) {
            if (r >= j.nv || r >= stream_end(j)) continue;
            if (r == 0 && fused0(j)) continue;
            const bool fuse = r == 1 && fused0(j);
            any_fused = any_fused || fuse;
            Node& n = *nodes_[j.node];
            Work& wb = wk(j);
            ProdItem<FP> it;
            it.nt = j.nt;
            if (r == 0) {
                it.w_in = weights(j); it.w_out = nullptr; it.tab_in = tables(n); it.tab_out = nullptr; it.n_in = j.S; it.r_prev = nullptr;
            } else {
                it.n_in = j.S >> (r - 1);
                it.w_in = r == 1 ? weights(j) : ((r - 1) & 1 ? wb.wbuf0.p : wb.wbuf1.p);
                it.w_out = (r & 1) ? wb.wbuf0.p : wb.wbuf1.p;
                it.tab_in = r == 1 ? (const void*)tables(n) : (const void*)((r - 1) & 1 ? wb.tbuf0.p : wb.tbuf1.p);
                it.tab_out = (r & 1) ? wb.tbuf0.p : wb.tbuf1.p;
                it.r_prev = ch.d_chal(j.r0_idx + r - 1);
            }
            it.msg = ch.d_msg(j.msg_off + 4 * (size_t)(fuse ? 0 : r));
            const size_t npairs = r == 0 ? it.n_in / 2 : it.n_in / 4;
            // several pairs per thread: the block-level reduction that ends every block costs about as much as eight pairs (measured optimum 8-16)
            constexpr size_t ppt_max = 16;
            const size_t ppt = std::max<size_t>(1, std::min<size_t>(ppt_max, round_pairs / ((size_t)HG_PROD_BLOCK * ctx_->sm_count * 4)));
            size_t b = std::max<size_t>(1, std::min<size_t>((npairs + HG_PROD_BLOCK * ppt - 1) / (HG_PROD_BLOCK * ppt), (size_t)ctx_->sm_count * 16 * (HG_BLOCK / HG_PROD_BLOCK)));
            it.nblk = (int)b; it.bx = (int)b; it.blk_start = blk;
            blk += it.nblk;
            it.partials = d_partials_.p + part_off;
            part_off += b * (fuse ? 8 : 4);
            it.counter = d_counters_.p + 8 + items.size();
            bytes += it.n_in * ((r <= 1 ? sizeof(B) : sizeof(X)) * j.nt + sizeof(X)) + (r ? (it.n_in / 2) * sizeof(X) * (j.nt + 1) : 0);
            items.push_back(it);
        }
        if (items.empty()) return;
        if (part_off > d_partials_.n) throw std::runtime_error("gkr: partial-sum pool too small");
        if (desc_off_ > h_desc_.n - (1 << 16)) { HG_CUDA(cudaStreamSynchronize(s)); desc_off_ = 0; }
        const ProdItem<FP>* di = stage(items);
        KernelScope ks(ctx_, KC_GKR_SC, bytes);
        if (r == 0) k_prod_round_multi<FP, B, false><<<blk, HG_PROD_BLOCK, 0, s>>>(di, (int)items.size());
        else if (r == 1 && any_fused) k_prod_round_multi<FP, B, true, true><<<blk, HG_PROD_BLOCK, 0, s>>>(di, (int)items.size());
        else if (r == 1) k_prod_round_multi<FP, B, true><<<blk, HG_PROD_BLOCK, 0, s>>>(di, (int)items.size());
        else k_prod_round_multi<FP, X, true><<<blk, HG_PROD_BLOCK, 0, s>>>(di, (int)items.size());
        HG_LAUNCH_CHECK();
        // linear layers: the table folded over the low log2(n_in) variables holds the evaluations of the inputs; it is the
        // output of round m = log2(n_in) and would be overwritten two rounds later, so it is copied out now
        std::vector<CopyItem<FP>> copies;
        for (const Job& j : jobs) {
            Node& n = *nodes_[j.node];
            Work& wb = wk(j);
            if (!lin(n)) continue;
            const int m = log2sz(n.n_in);
            if (m != r || m >= j.nv || r == 0 || m >= stream_end(j)) continue;
            CopyItem<FP> c; c.src = (m & 1) ? wb.tbuf0.p : wb.tbuf1.p; c.dst = wb.capture.p; c.n = n.arity;
            copies.push_back(c);
        }
        if (!copies.empty()) HG_K(ctx_, KC_GKR_SC, copies.size() * 64, k_copy_items<FP><<<(unsigned)copies.size(), 32, 0, s>>>(stage(copies)));
    }

    // first round that is NOT streamed: the tail kernel takes over there (prefetch mode only; nv when the job has no tail)
    // Round schedule of a job in prefetch mode (use_tail_): rounds [0, stream_end) are streamed, one launch per round for all jobs,
    // and the rest (tables of <= 2^10 entries) run in the one-CTA-per-job tail kernel. Without use_tail_ every round is streamed.
    int stream_end(const Job& j) const {
        if (!use_tail_ || j.nv < 3) return j.nv;
        return std::max(2, j.nv - HG_PROD_TAIL_LOG);
    }
    // rounds stream_end .. nv-1 and the input evaluations of every job that has a tail, one CTA per job
    void launch_tail(Channel<FP>& ch, const std::vector<Job>& jobs) {
        cudaStream_t s = ctx_->stream;
        std::vector<ProdTailItem<FP>> items;
        size_t smem = 0, bytes = 0;
        for (const Job& j : jobs) {
            const int rt = stream_end(j);
            if (rt >= j.nv) continue;
            Node& n = *nodes_[j.node];
            Work& wb = wk(j);
            ProdTailItem<FP> t;
            t.n_in = (int)(j.S >> (rt - 1)); t.nt = j.nt; t.rounds = j.nv - rt;
            t.w_in = ((rt - 1) & 1) ? wb.wbuf0.p : wb.wbuf1.p;
            t.tab_in = ((rt - 1) & 1) ? wb.tbuf0.p : wb.tbuf1.p;
            t.mid_part = nullptr; t.mid_msg = nullptr; t.mid_nseg = 0; t.mid_rounds = 0;
            t.chal = ch.d_chal(j.r0_idx + rt - 1);
            t.msg = ch.d_msg(j.msg_off + 4 * (size_t)rt);
            t.evals = ch.d_msg(j.evals_off);
            t.linear = lin(n);
            t.arity = n.arity; t.capture = nullptr; t.cap_round = -1;
            if (t.linear) {
                const int m = log2sz(n.n_in);
                if (m == 0) throw std::runtime_error("gkr: empty input tables");
                if (m < rt) t.capture = wb.capture.p;
                else if (m < j.nv) t.cap_round = m - rt;
            }
            smem = std::max(smem, ((size_t)(j.nt + 1) * (t.n_in + t.n_in / 2) + 96) * sizeof(X));
            bytes += (size_t)(j.nt + 1) * t.n_in * sizeof(X);
            items.push_back(t);
        }
        if (items.empty()) return;
        HG_K(ctx_, KC_GKR_SC, bytes, k_prod_tail<FP><<<(unsigned)items.size(), 256, smem, s>>>(stage(items)));
    }

    // input evaluations: linear layers read them off the table folded over the low variables; FFT / product layers off the last fold
    void launch_finals(Channel<FP>& ch, const std::vector<Job>& jobs) {
        cudaStream_t s = ctx_->stream;
        std::vector<FoldItem<FP>> folds;
        std::vector<CopyItem<FP>> copies;
        for (const Job& j : jobs) {
            if (stream_end(j) < j.nv) continue;  // done by launch_tail
            Node& n = *nodes_[j.node];
            Work& wb = wk(j);
            // state after the last round launch (round nv-1): tables folded by r_0..r_{nv-2}, length 2
            const int last = j.nv - 1;
            const void* tab_last = last == 0 ? (const void*)tables(n) : (const void*)((last & 1) ? wb.tbuf0.p : wb.tbuf1.p);
            const bool base_last = last == 0;
            if (lin(n)) {
                const int m = log2sz(n.n_in);  // the table folded by r_0..r_{m-1} has a_pad entries: the evaluations of the inputs
                if (m == j.nv) {
                    FoldItem<FP> f; f.in = tab_last; f.out = ch.d_msg(j.evals_off); f.r = ch.d_chal(j.r0_idx + j.nv - 1); f.n_out = 1; f.in_base = base_last;
                    folds.push_back(f);
                } else if (m == 0) {
                    throw std::runtime_error("gkr: empty input tables");
                } else {  // captured by launch_round(m) into the node's staging buffer
                    CopyItem<FP> c; c.src = wb.capture.p; c.dst = ch.d_msg(j.evals_off); c.n = n.arity;
                    copies.push_back(c);
                }
            } else {
                FoldItem<FP> f; f.in = tab_last; f.out = ch.d_msg(j.evals_off); f.r = ch.d_chal(j.r0_idx + j.nv - 1); f.n_out = j.nt; f.in_base = base_last;
                // nt tables of length 2 are contiguous: [t0_0 t0_1 t1_0 t1_1] -> out[q] = fold(in[2q], in[2q+1])
                folds.push_back(f);
            }
        }
        if (!folds.empty()) HG_K(ctx_, KC_GKR_SC, folds.size() * 64, k_fold_items<FP><<<(unsigned)folds.size(), 32, 0, s>>>(stage(folds)));
        if (!copies.empty()) HG_K(ctx_, KC_GKR_SC, copies.size() * 64, k_copy_items<FP><<<(unsigned)copies.size(), 32, 0, s>>>(stage(copies)));
    }

    double timing_[6] = {0, 0, 0, 0, 0, 0};
    DeviceCtx* ctx_;
    NttEngine<FP>* ntt_;
    std::vector<std::unique_ptr<Node>> nodes_;
    std::vector<int> topo_;
    bool evaluated_ = false, planned_ = false, eval_planned_ = false, use_tail_ = false;
    std::vector<EvalLevel> eval_levels_;
    size_t total_chal_ = 0, desc_off_ = 0, eq_off_ = 0;
    std::unique_ptr<Channel<FP>> ch_;
    DevBuf<X> d_eq_, d_partials_, d_outpts_;
    PinnedBuf<X> h_outpts_;
    DevBuf<B> d_planes_;
    DevBuf<unsigned> d_counters_;
    DevBuf<unsigned char> d_desc_;
    PinnedBuf<unsigned char> h_desc_;
};

}  // namespace hg
