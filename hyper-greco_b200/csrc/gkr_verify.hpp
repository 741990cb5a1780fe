// Host verifier of gkr::verify_gkr for the node shapes bfv-gkr builds: the other half of BfvEncrypt::verify
// (/root/reference/bfv-gkr/src/sk_encryption_circuit.rs:462-517; verify_gkr call at :509-510, input-claim check at :512-516).
// No CUDA, no device: a circuit DESCRIPTION (hg_circuit_new_host) is enough.
//
// The engine itself is the un-vendored `gkr` crate (PARITY UNPINNED, DESIGN.md section 3). This verifier checks exactly the protocol the
// device prover (gkr_dev.cuh) speaks, node by node in reverse topological order:
//     [T > 1 claims on the node: squeeze alpha]  ->  product sumcheck rounds (wire format A3)  ->  read the input evaluations
//     final check   W(r) * prod_k in_k(r) == last sumcheck claim,   W = the weights the claims induce on the node's inputs
//       Vanilla, additive gates   W = sum_t alpha^t eq(z_t, .) pushed through the wiring (plus the constant part of the gates)
//       element-wise product      W = sum_t alpha^t eq(z_t, .)
//       Vanilla, general gates    two product sumchecks (x, then y), final check X(u) M(u, v) X(v) == last claim (DESIGN.md section 3, A11)
//       FFT forward / inverse     W = transform of sum_t alpha^t eq(z_t, .)   (the DFT matrix is symmetric)
//       Lasso                     LassoVerifier (lasso_verify.hpp)
// It returns the claims that reach the input nodes; the caller compares them with the MLEs of the inputs (hg_mle_eval_host).
#pragma once
#include <algorithm>
#include <memory>

#include "gkr_dev.cuh"
#include "lasso_verify.hpp"

namespace hg {

// gkr::sum_check::verify_sum_check for a degree-`deg` round polynomial [UPSTREAM, assumptions A3 / A3']
template <class FP>
void verify_sum_check_host(int deg, int nv, typename FP::X claim, Keccak256Transcript<FP>& tr, const WireOptions& wo, typename FP::X* out_claim,
                           std::vector<typename FP::X>* out_point) {
    typedef typename FP::X X;
    typedef RoundPoly<FP> RP;
    out_point->clear();
    for (int j = 0; j < nv; j++) {
        std::vector<X> msg(deg);
        for (auto& v : msg) v = tr.read_felt_ext();
        std::vector<X> co(deg + 1);
        if (wo.a3_wire == 0) {
            co[0] = msg[0];
            X rest = FP::x_add(co[0], co[0]);
            for (int k = 2; k <= deg; k++) { co[k] = msg[k - 1]; rest = FP::x_add(rest, co[k]); }
            co[1] = FP::x_sub(claim, rest);
        } else {
            std::vector<X> ev(deg + 1);
            ev[0] = msg[0];
            ev[1] = FP::x_sub(claim, ev[0]);
            for (int k = 2; k <= deg; k++) ev[k] = msg[k - 1];
            co = RP::interpolate(ev);
        }
        const X rj = tr.squeeze_challenge();
        claim = RP::horner(co, rj);
        out_point->push_back(rj);
    }
    *out_claim = claim;
}

template <class FP> class GkrVerifierHost {
  public:
    typedef typename FP::B B;
    typedef typename FP::X X;
    struct Claim { std::vector<X> point; X value; };

    int insert_input(size_t log2_size, size_t num_reps) {
        Node n;
        n.kind = GKR_INPUT; n.out_len = num_reps << log2_size;
        nodes_.push_back(std::move(n));
        return (int)nodes_.size() - 1;
    }
    int insert_fft(size_t log2_size, bool inverse) {
        if (log2_size > (size_t)FP::TWO_ADICITY) throw VerifyError("FftNode: size exceeds the field's two-adicity");
        Node n;
        n.kind = GKR_FFT; n.out_len = (size_t)1 << log2_size; n.log2_size = (int)log2_size; n.fft_inverse = inverse;
        nodes_.push_back(std::move(n));
        return (int)nodes_.size() - 1;
    }
    int insert_lasso(const LassoPreprocessing& pp, int num_vars) {
        Node n;
        n.kind = GKR_LASSO; n.out_len = 1; n.pp.reset(new LassoPreprocessing(pp)); n.lasso_nv = num_vars;
        nodes_.push_back(std::move(n));
        return (int)nodes_.size() - 1;
    }
    int insert_vanilla(const VanillaDesc& d) {
        const size_t ng = d.n_gates, sub = (size_t)1 << d.log2_sub;
        if (d.arity < 1 || d.num_reps < 1 || ng < 1 || d.add_ptr.size() != ng + 1 || d.mul_ptr.size() != ng + 1 || d.has_const.size() != ng)
            throw VerifyError("VanillaNode: bad descriptor");
        const size_t n_add = d.add_ptr[ng], n_mul = d.mul_ptr[ng];
        for (size_t g = 0; g < ng; g++) if (d.add_ptr[g + 1] < d.add_ptr[g] || d.mul_ptr[g + 1] < d.mul_ptr[g]) throw VerifyError("VanillaNode: CSR pointers must be non-decreasing");
        for (size_t e = 0; e < n_add; e++) if (d.add_in[e] >= d.arity || d.add_wire[e] >= sub) throw VerifyError("VanillaNode: edge outside the inputs");
        for (size_t e = 0; e < n_mul; e++)
            if (d.mul_in0[e] >= d.arity || d.mul_in1[e] >= d.arity || d.mul_w0[e] >= sub || d.mul_w1[e] >= sub) throw VerifyError("VanillaNode: edge outside the inputs");
        Node n;
        n.kind = GKR_VANILLA; n.arity = (int)d.arity; n.log2_sub = (int)d.log2_sub; n.num_reps = (int)d.num_reps; n.ng = ng;
        n.out_len = pad2(ng * d.num_reps);
        n.n_in = d.num_reps << d.log2_sub;
        n.a_pad = pad2(d.arity);
        n.is_linear = n_mul == 0;
        if (!n.is_linear) {
            bool ok = d.arity == 2 && n_add == 0 && n_mul == ng && d.num_reps == 1;
            for (size_t g = 0; ok && g < ng; g++)
                ok = !d.has_const[g] && d.mul_ptr[g] == g && d.mul_in0[g] == 0 && d.mul_in1[g] == 1 && d.mul_w0[g] == g && d.mul_w1[g] == g &&
                     FP::b_eq(FP::b_from_limbs(&d.mul_coef[g * FP::B_LIMBS]), FP::b_one());
            n.is_elemmul = ok;  // otherwise a general layer (two-phase layer sumcheck)
        }
        if (!n.is_elemmul) n.desc.reset(new VanillaDesc(d));
        nodes_.push_back(std::move(n));
        return (int)nodes_.size() - 1;
    }
    void connect(int from, int to) {
        if (from < 0 || to < 0 || from >= (int)nodes_.size() || to >= (int)nodes_.size()) throw VerifyError("connect: no such node");
        nodes_[to].preds.push_back(from);
        nodes_[from].succs.push_back(to);
    }
    size_t num_nodes() const { return nodes_.size(); }

    // verify_gkr: one output claim per output node (insertion order); returns the claims on the input nodes (insertion order)
    std::vector<std::vector<Claim>> verify(Keccak256Transcript<FP>& tr, const WireOptions& wo, const std::vector<Claim>& output_claims) {
        std::vector<std::vector<Claim>> claims(nodes_.size());
        std::vector<int> outs;
        for (size_t i = 0; i < nodes_.size(); i++) if (nodes_[i].succs.empty() && nodes_[i].kind != GKR_INPUT) outs.push_back((int)i);
        if (outs.size() != output_claims.size()) throw VerifyError("verify_gkr: one output claim per output node is required");
        for (size_t i = 0; i < outs.size(); i++) claims[outs[i]].push_back(output_claims[i]);
        const std::vector<int> ord = topo();
        for (size_t oi = ord.size(); oi-- > 0;) {
            const int id = ord[oi];
            const Node& n = nodes_[id];
            if (n.kind == GKR_INPUT) continue;
            std::vector<std::vector<Claim>> sub = verify_node(n, claims[id], tr, wo);
            for (size_t k = 0; k < sub.size(); k++) for (auto& c : sub[k]) claims[n.preds.at(k)].push_back(c);
        }
        std::vector<std::vector<Claim>> res;
        for (size_t i = 0; i < nodes_.size(); i++) if (nodes_[i].kind == GKR_INPUT) res.push_back(claims[i]);
        return res;
    }

    // ---- host helpers shared with the C ABI
    // eq(point, i) for all i < 2^|point|, variable 0 = least significant bit (A4, A10)
    static std::vector<X> eq_table(const std::vector<X>& point) {
        std::vector<X> t(1, FP::x_one());
        t.reserve((size_t)1 << point.size());
        for (size_t k = 0; k < point.size(); k++) {
            const size_t half = t.size();
            t.resize(2 * half);
            const X one_minus = FP::x_sub(FP::x_one(), point[k]);
            for (size_t i = 0; i < half; i++) { const X v = t[i]; t[i] = FP::x_mul(v, one_minus); t[i + half] = FP::x_mul(v, point[k]); }
        }
        return t;
    }
    // multilinear extension of an extension-field table at `point` (length 2^|point|), by folding the lowest variable first
    static X mle_eval_ext(std::vector<X> t, const std::vector<X>& point) {
        if (t.size() != (size_t)1 << point.size()) throw VerifyError("mle_eval: table size does not match the point");
        size_t n = t.size();
        for (size_t k = 0; k < point.size(); k++) {
            n >>= 1;
            for (size_t i = 0; i < n; i++) t[i] = FP::x_add(t[2 * i], FP::x_mul(point[k], FP::x_sub(t[2 * i + 1], t[2 * i])));
        }
        return t[0];
    }
    static X mle_eval_base(const B* table, size_t len, const std::vector<X>& point) {
        if (len != (size_t)1 << point.size()) throw VerifyError("mle_eval: table size does not match the point");
        if (point.empty()) return FP::lift(table[0]);
        std::vector<X> t(len / 2);
        for (size_t i = 0; i < len / 2; i++) t[i] = FP::x_add(FP::lift(table[2 * i]), FP::x_mul_b(point[0], FP::b_sub(table[2 * i + 1], table[2 * i])));
        return mle_eval_ext(std::move(t), std::vector<X>(point.begin() + 1, point.end()));
    }
    // radix-2 NTT, natural order in and out, w = ROOT_OF_UNITY^(2^(S - log n)); inverse scaled by 1/n (A9)
    static void ntt_host(std::vector<B>& a, bool inverse) {
        const size_t n = a.size();
        int lg = 0;
        while (((size_t)1 << lg) < n) lg++;
        if (((size_t)1 << lg) != n || lg > FP::TWO_ADICITY) throw VerifyError("ntt: bad size");
        for (size_t i = 1, j = 0; i < n; i++) {
            size_t bit = n >> 1;
            for (; j & bit; bit >>= 1) j ^= bit;
            j ^= bit;
            if (i < j) std::swap(a[i], a[j]);
        }
        B w = FP::root_of_unity();
        for (int k = lg; k < FP::TWO_ADICITY; k++) w = FP::b_mul(w, w);
        if (inverse) w = FP::b_inv(w);
        std::vector<B> tw(std::max<size_t>(n / 2, 1));
        tw[0] = FP::b_one();
        for (size_t i = 1; i < n / 2; i++) tw[i] = FP::b_mul(tw[i - 1], w);
        for (size_t len = 2; len <= n; len <<= 1) {
            const size_t step = n / len, half = len / 2;
            for (size_t s = 0; s < n; s += len)
                for (size_t k = 0; k < half; k++) {
                    const B u = a[s + k], v = FP::b_mul(a[s + k + half], tw[k * step]);
                    a[s + k] = FP::b_add(u, v);
                    a[s + k + half] = FP::b_sub(u, v);
                }
        }
        if (inverse) {
            const B ninv = FP::b_inv(FP::b_from_u64((u64)n));
            for (auto& v : a) v = FP::b_mul(v, ninv);
        }
    }

  private:
    struct Node {
        int kind = GKR_INPUT, log2_size = 0, num_reps = 1, arity = 0, log2_sub = 0, lasso_nv = 0;
        bool fft_inverse = false, is_linear = false, is_elemmul = false;
        size_t ng = 0, out_len = 0, n_in = 0, a_pad = 1;
        std::vector<int> preds, succs;
        std::shared_ptr<VanillaDesc> desc;            // linear and general layers: the gates (CSR)
        std::shared_ptr<LassoPreprocessing> pp;
    };
    static size_t pad2(size_t n) { size_t p = 1; while (p < n) p <<= 1; return p; }
    static int log2sz(size_t n) { int l = 0; while (((size_t)1 << l) < n) l++; return l; }

    std::vector<int> topo() const {  // Kahn, always the ready node with the smallest insertion index (as the prover)
        std::vector<int> indeg(nodes_.size()), order;
        std::vector<char> done(nodes_.size(), 0);
        for (size_t i = 0; i < nodes_.size(); i++) indeg[i] = (int)nodes_[i].preds.size();
        for (size_t step = 0; step < nodes_.size(); step++) {
            int pick = -1;
            for (size_t i = 0; i < nodes_.size(); i++) if (!done[i] && indeg[i] == 0) { pick = (int)i; break; }
            if (pick < 0) throw VerifyError("circuit has a cycle");
            done[pick] = 1; order.push_back(pick);
            for (int sx : nodes_[pick].succs) indeg[sx]--;
        }
        return order;
    }

    std::vector<std::vector<Claim>> verify_node(const Node& n, const std::vector<Claim>& cl, Keccak256Transcript<FP>& tr, const WireOptions& wo) {
        std::vector<std::vector<Claim>> out(n.preds.size());
        if (n.kind == GKR_LASSO) {
            if (n.preds.size() != 1) throw VerifyError("the Lasso node takes exactly one input (lasso.rs:64)");
            LassoVerifier<FP> lv(*n.pp, n.lasso_nv, wo);
            Claim c;
            lv.verify(tr, &c.point, &c.value);
            out[0].push_back(c);
            return out;
        }
        if (cl.empty()) throw VerifyError("verify_gkr: node without claims");
        X alpha = FP::x_one();
        if (cl.size() > 1) alpha = tr.squeeze_challenge();
        // combined claim and W = sum_t alpha^t eq(z_t, .)
        X combined = FP::x_zero();
        std::vector<X> w(n.out_len, FP::x_zero());
        {
            X p = FP::x_one();
            for (auto& c : cl) {
                if (((size_t)1 << c.point.size()) != n.out_len) throw VerifyError("verify_gkr: claim point does not match the node's output size");
                combined = FP::x_add(combined, FP::x_mul(p, c.value));
                const std::vector<X> eq = eq_table(c.point);
                for (size_t i = 0; i < n.out_len; i++) w[i] = FP::x_add(w[i], FP::x_mul(p, eq[i]));
                p = FP::x_mul(p, alpha);
            }
        }
        std::vector<X> pt;
        X fc;
        if (n.kind == GKR_FFT) {
            verify_sum_check_host<FP>(2, n.log2_size, combined, tr, wo, &fc, &pt);
            const X in_eval = tr.read_felt_ext();
            // A = transform(W), plane by plane
            std::vector<B> plane(n.out_len);
            std::vector<X> A(n.out_len);
            std::vector<B> planes[4];
            for (int q = 0; q < FP::PLANES; q++) {
                for (size_t i = 0; i < n.out_len; i++) plane[i] = FP::plane(w[i], q);
                ntt_host(plane, n.fft_inverse);
                planes[q] = plane;
            }
            for (size_t i = 0; i < n.out_len; i++) {
                B b[4];
                for (int q = 0; q < FP::PLANES; q++) b[q] = planes[q][i];
                A[i] = FP::from_planes(b);
            }
            if (!FP::x_eq(FP::x_mul(mle_eval_ext(std::move(A), pt), in_eval), fc)) throw VerifyError("InvalidSumCheck: FFT layer final evaluation mismatch");
            out.at(0).push_back({pt, in_eval});
        } else if (n.is_elemmul) {
            verify_sum_check_host<FP>(3, log2sz(n.out_len), combined, tr, wo, &fc, &pt);
            const X a = tr.read_felt_ext(), b = tr.read_felt_ext();
            if (!FP::x_eq(FP::x_mul(FP::x_mul(mle_eval_ext(std::move(w), pt), a), b), fc)) throw VerifyError("InvalidSumCheck: product layer final evaluation mismatch");
            out.at(0).push_back({pt, a});
            out.at(1).push_back({pt, b});
        } else if (n.is_linear) {
            if ((int)n.preds.size() != n.arity) throw VerifyError("Vanilla node arity does not match its connections");
            const VanillaDesc& d = *n.desc;
            const size_t S = n.a_pad * n.n_in, sub = (size_t)1 << n.log2_sub;
            std::vector<X> A(S, FP::x_zero());
            X constant = FP::x_zero();
            for (size_t r = 0; r < (size_t)n.num_reps; r++)
                for (size_t g = 0; g < n.ng; g++) {
                    const X wg = w[r * n.ng + g];
                    if (d.has_const[g]) constant = FP::x_add(constant, FP::x_mul_b(wg, FP::b_from_limbs(&d.consts[g * FP::B_LIMBS])));
                    for (uint64_t e = d.add_ptr[g]; e < d.add_ptr[g + 1]; e++) {
                        X& a = A[(size_t)d.add_in[e] * n.n_in + r * sub + d.add_wire[e]];
                        a = FP::x_add(a, FP::x_mul_b(wg, FP::b_from_limbs(&d.add_coef[e * FP::B_LIMBS])));
                    }
                }
            verify_sum_check_host<FP>(2, log2sz(S), FP::x_sub(combined, constant), tr, wo, &fc, &pt);
            const int lo_vars = log2sz(n.n_in);
            std::vector<X> lo(pt.begin(), pt.begin() + lo_vars), hi(pt.begin() + lo_vars, pt.end());
            const std::vector<X> eqhi = eq_table(hi);
            X x = FP::x_zero();
            for (int k = 0; k < n.arity; k++) {
                const X e = tr.read_felt_ext();
                x = FP::x_add(x, FP::x_mul(eqhi[k], e));
                out[k].push_back({lo, e});
            }
            if (!FP::x_eq(FP::x_mul(mle_eval_ext(std::move(A), pt), x), fc)) throw VerifyError("InvalidSumCheck: linear layer final evaluation mismatch");
        } else {  // general layer: phase 1 over x (claim c - const), phase 2 over y (claim fc1 - A(u) X(u)), DESIGN.md section 3 (A11)
            if ((int)n.preds.size() != n.arity) throw VerifyError("Vanilla node arity does not match its connections");
            const VanillaDesc& d = *n.desc;
            const size_t S = n.a_pad * n.n_in, sub = (size_t)1 << n.log2_sub;
            const int nv = log2sz(S), lo_vars = log2sz(n.n_in);
            X constant = FP::x_zero();
            for (size_t r = 0; r < (size_t)n.num_reps; r++)
                for (size_t g = 0; g < n.ng; g++)
                    if (d.has_const[g]) constant = FP::x_add(constant, FP::x_mul_b(w[r * n.ng + g], FP::b_from_limbs(&d.consts[g * FP::B_LIMBS])));
            auto read_evals = [&](const std::vector<X>& p) {  // X(p) = sum_k eq(p_hi, k) X_k(p_lo) from the written X_k(p_lo)
                const std::vector<X> lo(p.begin(), p.begin() + lo_vars), hi(p.begin() + lo_vars, p.end());
                const std::vector<X> eqhi = eq_table(hi);
                X x = FP::x_zero();
                for (int k = 0; k < n.arity; k++) {
                    const X e = tr.read_felt_ext();
                    x = FP::x_add(x, FP::x_mul(eqhi[k], e));
                    out[k].push_back({lo, e});
                }
                return x;
            };
            std::vector<X> u, v;
            X fc1, fc2;
            verify_sum_check_host<FP>(2, nv, FP::x_sub(combined, constant), tr, wo, &fc1, &u);
            const X xu = read_evals(u);
            const std::vector<X> equ = eq_table(u);
            // A(u) and M(u, v), sparsely from the edges
            X au = FP::x_zero();
            for (size_t r = 0; r < (size_t)n.num_reps; r++)
                for (size_t g = 0; g < n.ng; g++)
                    for (uint64_t e = d.add_ptr[g]; e < d.add_ptr[g + 1]; e++) {
                        const size_t x = (size_t)d.add_in[e] * n.n_in + r * sub + d.add_wire[e];
                        au = FP::x_add(au, FP::x_mul_b(FP::x_mul(w[r * n.ng + g], equ[x]), FP::b_from_limbs(&d.add_coef[e * FP::B_LIMBS])));
                    }
            verify_sum_check_host<FP>(2, nv, FP::x_sub(fc1, FP::x_mul(au, xu)), tr, wo, &fc2, &v);
            const X xv = read_evals(v);
            const std::vector<X> eqv = eq_table(v);
            X muv = FP::x_zero();
            for (size_t r = 0; r < (size_t)n.num_reps; r++)
                for (size_t g = 0; g < n.ng; g++)
                    for (uint64_t e = d.mul_ptr[g]; e < d.mul_ptr[g + 1]; e++) {
                        const size_t x = (size_t)d.mul_in0[e] * n.n_in + r * sub + d.mul_w0[e], y = (size_t)d.mul_in1[e] * n.n_in + r * sub + d.mul_w1[e];
                        muv = FP::x_add(muv, FP::x_mul_b(FP::x_mul(w[r * n.ng + g], FP::x_mul(equ[x], eqv[y])), FP::b_from_limbs(&d.mul_coef[e * FP::B_LIMBS])));
                    }
            if (!FP::x_eq(FP::x_mul(FP::x_mul(xu, muv), xv), fc2)) throw VerifyError("InvalidSumCheck: general layer final evaluation mismatch");
        }
        return out;
    }

    std::vector<Node> nodes_;
};

}  // namespace hg
