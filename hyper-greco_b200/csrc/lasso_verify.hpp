// Host verifier of the Lasso node: Node::verify_claim_reduction (/root/reference/lasso/src/lasso.rs:116-139), with
// MemoryCheckingVerifier::verify (/root/reference/lasso/src/memory_checking/verifier.rs:130-176), verify_grand_product
// (:178-235) and Chunk::verify_memories (:61-95). Field-generic over the same policies as the kernels (host functions only);
// no CUDA. The sumcheck message format is the upstream `gkr` crate's (not vendored): the WireOptions switches of prover.cuh
// apply here as well. Subtable MLEs are evaluated from the materialised tables (the MLE is unique, so this equals the
// reference's closed forms, table/range.rs:28-38,114-161).
#pragma once
#include <map>
#include <stdexcept>
#include <string>
#include <vector>

#include "prover.cuh"

namespace hg {

struct VerifyError : std::runtime_error {
    explicit VerifyError(const std::string& m) : std::runtime_error(m) {}
};

// A final check of the replay left to the device: coef[0] q[0] + coef[1] q[1] + coef[2] q[2] == target, where the q[j] are
// linear-size quantities of the circuit fixed by the claim points, alpha, pt and v (a coefficient is zero where the kind has no q[j]).
//   DC_FFT       q[0] = MLE(transform(W))(pt),  W = sum_t alpha^t eq(z_t, .) over the node's outputs
//   DC_LINEAR    q[0] = MLE(A)(pt), A = W pushed through the additive edges; q[1] = sum_g W[g] const_g (the claim's constant part)
//   DC_GENERAL   q[0] = A(pt) and q[1] as for DC_LINEAR, q[2] = M(pt, v) = sum over the product edges of coef W[out] eq(pt, x) eq(v, y)
//   DC_SUBTABLE  q[0] = MLE(subtable `index`)(pt)
//   DC_INPUT     q[0] = MLE(input node `index`)(pt)
enum DeferredKind { DC_FFT = 0, DC_LINEAR, DC_SUBTABLE, DC_INPUT, DC_GENERAL };
template <class FP> struct DeferredCheck {
    typedef typename FP::X X;
    int kind = DC_FFT, index = 0;  // node id (FFT, linear, general), subtable index, input index
    std::vector<std::vector<X>> z;  // claim points (FFT, linear, general)
    X alpha, target;
    X coef[3] = {FP::x_zero(), FP::x_zero(), FP::x_zero()};
    std::vector<X> pt, v;           // v: the general layer's phase-2 point
    const char* what = "";          // the rejection reason when the equality fails
};
template <class FP> using DeferredChecks = std::vector<DeferredCheck<FP>>;

template <class FP> class LassoVerifier {
  public:
    typedef typename FP::B B;
    typedef typename FP::X X;
    LassoVerifier(const LassoPreprocessing& pp, int num_vars, const WireOptions& wo) : pp_(pp), num_vars_(num_vars), wo_(wo) {
        log2M_ = (int)ilog2u(pp.M);
        std::map<size_t, std::vector<size_t>> by_dim;  // chunks: memories grouped by dimension, ascending (lasso.rs:303-336)
        for (size_t mi = 0; mi < pp.num_memories; mi++) by_dim[pp.memory_to_dimension_index[mi]].push_back(mi);
        for (auto& kv : by_dim) chunks_.push_back(kv.second);
    }

    // reads the node's part of the proof from `tr`, squeezing the challenges the prover squeezed; returns (r, claimed_sum).
    // With `defer`, the init_ys / final_read_ys equalities, the only use of the subtable values st_y, become records
    // gamma * st_y == ify - id_y - t gamma^2 + tau (DC_SUBTABLE) instead of materialising the subtables here.
    void verify(Keccak256Transcript<FP>& tr, std::vector<X>* out_r, X* out_claimed_sum, DeferredChecks<FP>* defer = nullptr) {
        std::vector<X> r(num_vars_);
        for (auto& c : r) c = tr.squeeze_challenge();                         // lasso.rs:123
        const X claimed_sum = tr.read_felt_ext();                             // lasso.rs:344
        { X fin; std::vector<X> pt; verify_sum_check(2, num_vars_, claimed_sum, tr, &fin, &pt); }  // result unused: lasso.rs:129-133
        const X gamma_e = tr.squeeze_challenge(), tau_e = tr.squeeze_challenge();   // lasso.rs:135
        const B gamma = FP::x_base0(gamma_e), tau = FP::x_base0(tau_e), gamma2 = FP::b_mul(gamma, gamma);   // verifier.rs:139-140
        const size_t m = pp_.num_memories;
        std::vector<X> rw, x, ify, y;
        verify_grand_product(num_vars_, 2 * m, tr, &rw, &x);                  // verifier.rs:143-150
        verify_grand_product(log2M_, 2 * m, tr, &ify, &y);
        auto hash = [&](X a, X v, X t) {                                       // verifier.rs:158: a + v*gamma + t*gamma^2 - tau
            return FP::x_sub(FP::x_add(FP::x_add(a, FP::x_mul_b(v, gamma)), FP::x_mul_b(t, gamma2)), FP::lift(tau));
        };
        X id_y = FP::x_zero();                                                // verifier.rs:74-78: sum_i 2^i y_i
        { X p2 = FP::x_one(); for (auto& yi : y) { id_y = FP::x_add(id_y, FP::x_mul(p2, yi)); p2 = FP::x_add(p2, p2); } }
        const std::vector<X> eq_y = defer ? std::vector<X>() : eq_table(y);
        std::map<size_t, X> subtable_at_y;                                     // LassoSubtable::evaluate_mle(y), one per subtable in use
        size_t off = 0;
        for (auto& mems : chunks_) {                                           // verifier.rs:61-95
            const X dim_x = tr.read_felt_ext(), ts_x = tr.read_felt_ext(), fc_y = tr.read_felt_ext();
            std::vector<X> e_x(mems.size());
            for (auto& e : e_x) e = tr.read_felt_ext();
            for (size_t i = 0; i < mems.size(); i++) {
                if (!FP::x_eq(rw[off + i], hash(dim_x, e_x[i], ts_x))) throw VerifyError("verify_memories: read_xs mismatch");
                if (!FP::x_eq(rw[m + off + i], hash(dim_x, e_x[i], FP::x_add(ts_x, FP::x_one())))) throw VerifyError("verify_memories: write_xs mismatch");
                const size_t st = pp_.memory_to_subtable_index[mems[i]];
                if (defer) {
                    for (int fin = 0; fin < 2; fin++) {
                        DeferredCheck<FP> d;
                        d.kind = DC_SUBTABLE; d.index = (int)st; d.pt = y; d.coef[0] = FP::lift(gamma);
                        const X t = fin ? fc_y : FP::x_zero();
                        d.target = FP::x_add(FP::x_sub(FP::x_sub(ify[(fin ? m : 0) + off + i], id_y), FP::x_mul_b(t, gamma2)), FP::lift(tau));
                        d.what = fin ? "verify_memories: final_read_ys mismatch" : "verify_memories: init_ys mismatch";
                        defer->push_back(std::move(d));
                    }
                    continue;
                }
                if (!subtable_at_y.count(st)) subtable_at_y[st] = table_mle(pp_.subtables_by_idx[st]->materialize(pp_.M), eq_y);
                const X st_y = subtable_at_y[st];
                if (!FP::x_eq(ify[off + i], hash(id_y, st_y, FP::x_zero()))) throw VerifyError("verify_memories: init_ys mismatch");
                if (!FP::x_eq(ify[m + off + i], hash(id_y, st_y, fc_y))) throw VerifyError("verify_memories: final_read_ys mismatch");
            }
            off += mems.size();
        }
        *out_r = r;
        *out_claimed_sum = claimed_sum;
    }

  private:
    // gkr::sum_check::verify_sum_check for a degree-`deg` function [UPSTREAM, assumptions A3/A3']: per round the message is
    // (c0, c2..cd) with c1 from h(0) + h(1) = claim, or the evaluations h(0), h(2)..h(d) with h(1) = claim - h(0)
    void verify_sum_check(int deg, int nv, X claim, Keccak256Transcript<FP>& tr, X* out_claim, std::vector<X>* out_point) {
        typedef RoundPoly<FP> RP;
        out_point->clear();
        for (int j = 0; j < nv; j++) {
            std::vector<X> msg(deg);
            for (auto& v : msg) v = tr.read_felt_ext();
            std::vector<X> co(deg + 1);
            if (wo_.a3_wire == 0) {
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
    // verifier.rs:178-235
    void verify_grand_product(int nv_gp, size_t nb, Keccak256Transcript<FP>& tr, std::vector<X>* out_claims, std::vector<X>* out_x) {
        std::vector<X> claimed(nb), evals(2 * nb), x;
        for (auto& c : claimed) c = tr.read_felt_ext();
        for (int nv = 0; nv < nv_gp; nv++) {
            if (nv == 0) {
                for (auto& e : evals) e = tr.read_felt_ext();
                for (size_t i = 0; i < nb; i++)
                    if (!FP::x_eq(claimed[i], FP::x_mul(evals[2 * i], evals[2 * i + 1]))) throw VerifyError("InvalidSumCheck: unmatched sum check output");
                x.clear();
            } else {
                const X gamma = tr.squeeze_challenge();
                X claim = FP::x_zero(), p = FP::x_one();
                for (size_t i = 0; i < nb; i++) { claim = FP::x_add(claim, FP::x_mul(claimed[i], p)); p = FP::x_mul(p, gamma); }
                X fin;
                verify_sum_check(3, nv, claim, tr, &fin, &x);  // the final claim is discarded (verifier.rs:218-221)
                for (auto& e : evals) e = tr.read_felt_ext();
            }
            const X mu = tr.squeeze_challenge();
            for (size_t i = 0; i < nb; i++) claimed[i] = FP::x_add(evals[2 * i], FP::x_mul(mu, FP::x_sub(evals[2 * i + 1], evals[2 * i])));
            x.push_back(mu);
        }
        *out_claims = claimed;
        *out_x = x;
    }
    // eq(y, i) for all i < 2^|y|, variable 0 = least significant bit (A4)
    static std::vector<X> eq_table(const std::vector<X>& y) {
        std::vector<X> t(1, FP::x_one());
        for (size_t k = 0; k < y.size(); k++) {
            const size_t half = t.size();
            t.resize(2 * half);
            const X one_minus = FP::x_sub(FP::x_one(), y[k]);
            for (size_t i = 0; i < half; i++) { const X v = t[i]; t[i] = FP::x_mul(v, one_minus); t[i + half] = FP::x_mul(v, y[k]); }
        }
        return t;
    }
    static X table_mle(const std::vector<uint64_t>& table, const std::vector<X>& eq) {
        if (table.size() != eq.size()) throw VerifyError("subtable size does not match the point");
        X acc = FP::x_zero();
        for (size_t i = 0; i < table.size(); i++) if (table[i]) acc = FP::x_add(acc, FP::x_mul_b(eq[i], FP::b_from_u64(table[i])));
        return acc;
    }

    const LassoPreprocessing& pp_;
    int num_vars_, log2M_ = 16;
    WireOptions wo_;
    std::vector<std::vector<size_t>> chunks_;
};

}  // namespace hg
