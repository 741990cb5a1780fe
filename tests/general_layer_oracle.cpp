// TEST INFRASTRUCTURE ONLY (tests/test_general_layer.py compiles it with g++ next to the oracle; the product never links it).
// An independent CPU restatement of general Vanilla layers: any layer with a product term other than the element-wise shape
// out[i] = in0[i] * in1[i] over every input wire (num_reps 1). It follows Libra's two-phase layer sumcheck as DESIGN.md section 7b states it
// (assumption A11) and reuses the oracle (oracle/gkr.hpp) for every other node shape, the transcript and the sumcheck.
// A C entry builds a generic circuit node by node: insert input / vanilla (the CSR of hg_circuit_insert_vanilla) / fft, connect,
// evaluate, prove_gkr, verify_gkr, for both fields.
#include <cstring>
#include <string>

#include "gkr.hpp"

using namespace hgo;

namespace {
thread_local std::string g_err;
template <class F> std::vector<F> load_base(const uint64_t* p, size_t n) {
    std::vector<F> v(n);
    for (size_t i = 0; i < n; i++) v[i] = F::from_limbs(p + i * F::LIMBS);
    return v;
}
template <class F, class E> E load_ext(const uint64_t* p) {
    F b[2];
    for (int i = 0; i < E::DEGREE; i++) b[i] = F::from_limbs(p + i * F::LIMBS);
    return E::from_bases(b);
}
template <class F, class E> void store_ext(const E& e, uint64_t* p) {
    F b[2]; e.as_bases(b);
    for (int i = 0; i < E::DEGREE; i++) b[i].to_limbs(p + i * F::LIMBS);
}

// the walk of prove_gkr / verify_gkr (oracle/gkr.hpp) with general layers proved here and every other node by the oracle
template <class F> struct GeneralCircuit {
    typedef typename ExtOf<F>::type E;
    typedef hgo::Circuit<F> C;
    C c;

    bool general(const GkrNode<F>& nd) const { return nd.kind == NODE_VANILLA && !nd.linear() && !nd.elementwise_mul(); }
    // fn(output index, coefficient, x, y) for every gate, rep and product term; x = (in0, r sub + w0), y = (in1, r sub + w1)
    // are positions in the concatenated inputs
    template <class Fn> static void for_each_product(const GkrNode<F>& nd, size_t n_in, Fn fn) {
        const size_t ng = nd.gates.size(), sub = (size_t)1 << nd.log2_sub_input;
        for (int r = 0; r < nd.num_reps; r++)
            for (size_t g = 0; g < ng; g++)
                for (auto& m : nd.gates[g].muls)
                    fn(r * ng + g, std::get<0>(m), (size_t)std::get<1>(m) * n_in + r * sub + std::get<2>(m), (size_t)std::get<3>(m) * n_in + r * sub + std::get<4>(m));
    }
    // [T > 1 claims: squeeze alpha], combined claim and w = sum_t alpha^t eq(z_t, .)
    static void combine(const GkrNode<F>& nd, const std::vector<EvalClaim<F>>& claims, Transcript<F>& tr, E* combined, std::vector<E>* w) {
        E alpha = E::one();
        if (claims.size() > 1) alpha = tr.squeeze();
        *combined = E::zero();
        E p = E::one();
        for (auto& cl : claims) { *combined += p * cl.value; p *= alpha; }
        *w = C::combined_eq(claims, alpha, nd.out_len());
    }

    std::vector<std::vector<EvalClaim<F>>> prove_general(int id, const std::vector<EvalClaim<F>>& claims, const std::vector<std::vector<F>>& val,
                                                         Transcript<F>& tr) const {
        const auto& nd = c.nodes[id];
        std::vector<std::vector<EvalClaim<F>>> out(nd.preds.size());
        E combined;
        std::vector<E> w;
        combine(nd, claims, tr, &combined, &w);
        typename C::Reduction R = c.linear_reduction(nd, w, &val);
        const std::vector<E> Xe = C::lift_vec(R.X);
        // phase 1 over x: G = A + H,  H[x] = sum_y M[x, y] X[y],  claim c - const
        std::vector<E> G = R.A, u, fin, cap;
        for_each_product(nd, R.n_in, [&](size_t o, const F& cf, size_t x, size_t y) { G[x] += w[o] * E::from_base(cf) * Xe[y]; });
        C::product_sumcheck({G, Xe}, combined - R.constant, tr, &u, &fin, R.a_pad, &cap, 1);
        const int m = C::log2sz(R.n_in);
        const std::vector<E> ulo(u.begin(), u.begin() + m);
        for (int k = 0; k < nd.arity; k++) { tr.write(cap[k]); out[k].push_back({ulo, cap[k]}); }
        // phase 2 over y: sum_y (X(u) M(u, y)) X(y) = fc1 - A(u) X(u), fc1 = G(u) X(u) the final claim of phase 1
        const E xu = fin[1], claim2 = fin[0] * fin[1] - mle_evaluate_ext(R.A, u) * xu;
        const std::vector<E> equ = eq_xy(u);
        std::vector<E> Mu(R.A.size(), E::zero()), v, cap2;
        for_each_product(nd, R.n_in, [&](size_t o, const F& cf, size_t x, size_t y) { Mu[y] += equ[x] * w[o] * E::from_base(cf); });
        for (auto& e : Mu) e = e * xu;
        C::product_sumcheck({Mu, Xe}, claim2, tr, &v, &fin, R.a_pad, &cap2, 1);
        const std::vector<E> vlo(v.begin(), v.begin() + m);
        for (int k = 0; k < nd.arity; k++) { tr.write(cap2[k]); out[k].push_back({vlo, cap2[k]}); }
        return out;
    }
    std::vector<std::vector<EvalClaim<F>>> verify_general(int id, const std::vector<EvalClaim<F>>& claims, Transcript<F>& tr) const {
        const auto& nd = c.nodes[id];
        std::vector<std::vector<EvalClaim<F>>> out(nd.preds.size());
        E combined;
        std::vector<E> w;
        combine(nd, claims, tr, &combined, &w);
        typename C::Reduction R = c.linear_reduction(nd, w, nullptr);
        const int nv = C::log2sz(R.a_pad * R.n_in), m = C::log2sz(R.n_in);
        auto read_evals = [&](const std::vector<E>& p) {  // X(p) = sum_k eq(p_hi, k) X_k(p_lo), from the written X_k(p_lo)
            const std::vector<E> lo(p.begin(), p.begin() + m), hi(p.begin() + m, p.end());
            const std::vector<E> eqhi = eq_xy(hi);
            E x = E::zero();
            for (int k = 0; k < nd.arity; k++) { E e = tr.read(); x += eqhi[k] * e; out[k].push_back({lo, e}); }
            return x;
        };
        std::vector<E> u, v;
        E fc1, fc2;
        C::product_sumcheck_verify(2, nv, combined - R.constant, tr, &u, &fc1);
        const E xu = read_evals(u);
        C::product_sumcheck_verify(2, nv, fc1 - mle_evaluate_ext(R.A, u) * xu, tr, &v, &fc2);
        const E xv = read_evals(v);
        const std::vector<E> equ = eq_xy(u), eqv = eq_xy(v);
        E muv = E::zero();
        for_each_product(nd, R.n_in, [&](size_t o, const F& cf, size_t x, size_t y) { muv += w[o] * E::from_base(cf) * equ[x] * eqv[y]; });
        if (xu * muv * xv != fc2) throw OracleError("InvalidSumCheck: general layer final evaluation mismatch");
        return out;
    }

    template <class Step> std::vector<std::vector<EvalClaim<F>>> walk(const std::vector<EvalClaim<F>>& output_claims, Step step) const {
        std::vector<std::vector<EvalClaim<F>>> claims(c.nodes.size());
        auto outs = c.output_nodes();
        if (outs.size() != output_claims.size()) throw OracleError("prove_gkr: output claim count mismatch");
        for (size_t i = 0; i < outs.size(); i++) claims[outs[i]].push_back(output_claims[i]);
        auto order = c.topo_order();
        for (size_t oi = order.size(); oi-- > 0;) {
            const int id = order[oi];
            if (c.nodes[id].kind == NODE_INPUT) continue;
            auto sub = step(id, claims[id]);
            for (size_t k = 0; k < sub.size(); k++) for (auto& cl : sub[k]) claims[c.nodes[id].preds[k]].push_back(cl);
        }
        std::vector<std::vector<EvalClaim<F>>> r;
        for (size_t id = 0; id < c.nodes.size(); id++) if (c.nodes[id].kind == NODE_INPUT) r.push_back(claims[id]);
        return r;
    }
    std::vector<std::vector<EvalClaim<F>>> prove_gkr(const std::vector<std::vector<F>>& val, const std::vector<EvalClaim<F>>& oc, Transcript<F>& tr) const {
        return walk(oc, [&](int id, const std::vector<EvalClaim<F>>& cl) { return general(c.nodes[id]) ? prove_general(id, cl, val, tr) : c.prove_node(id, cl, val, tr); });
    }
    std::vector<std::vector<EvalClaim<F>>> verify_gkr(const std::vector<EvalClaim<F>>& oc, Transcript<F>& tr) const {
        return walk(oc, [&](int id, const std::vector<EvalClaim<F>>& cl) { return general(c.nodes[id]) ? verify_general(id, cl, tr) : c.verify_node(id, cl, tr); });
    }
};

struct Session {
    virtual ~Session() {}
    virtual int insert_input(int log2_size, int reps) = 0;
    virtual int insert_fft(int log2_size, bool inverse) = 0;
    virtual int insert_vanilla(int arity, int log2_sub, int reps, size_t ng, const uint8_t* has_const, const uint64_t* consts, const uint64_t* add_ptr,
                               const uint64_t* add_coef, const uint32_t* add_in, const uint64_t* add_wire, const uint64_t* mul_ptr, const uint64_t* mul_coef,
                               const uint32_t* mul_in0, const uint64_t* mul_w0, const uint32_t* mul_in1, const uint64_t* mul_w1) = 0;
    virtual void connect(int from, int to) = 0;
    virtual void evaluate(const uint64_t* inputs) = 0;
    virtual size_t value(int id, uint64_t* out) = 0;
    virtual size_t prove(size_t n, const size_t* lens, const uint64_t* pts, const uint64_t* vals, uint8_t* proof, size_t cap) = 0;
    virtual void verify(size_t n, const size_t* lens, const uint64_t* pts, const uint64_t* vals, const uint8_t* proof, size_t len) = 0;
    virtual size_t num_inputs() const = 0;
    virtual size_t num_claims(size_t input) const = 0;
    virtual size_t claim(size_t input, size_t k, uint64_t* point, uint64_t* value) const = 0;
};
template <class F> struct SessionT : Session {
    typedef typename ExtOf<F>::type E;
    static constexpr size_t EL = E::DEGREE * F::LIMBS;
    GeneralCircuit<F> g;
    std::vector<std::vector<F>> val;
    std::vector<std::vector<EvalClaim<F>>> claims;
    static void check_reps(int reps) { if (reps < 1 || (reps & (reps - 1)) != 0) throw OracleError("num_reps must be a power of two"); }
    int insert_input(int log2_size, int reps) override { check_reps(reps); return g.c.insert(BfvEncrypt<F>::input(log2_size, reps)); }
    int insert_fft(int log2_size, bool inverse) override { return g.c.insert(BfvEncrypt<F>::fft(log2_size, inverse)); }
    int insert_vanilla(int arity, int log2_sub, int reps, size_t ng, const uint8_t* has_const, const uint64_t* consts, const uint64_t* add_ptr,
                       const uint64_t* add_coef, const uint32_t* add_in, const uint64_t* add_wire, const uint64_t* mul_ptr, const uint64_t* mul_coef,
                       const uint32_t* mul_in0, const uint64_t* mul_w0, const uint32_t* mul_in1, const uint64_t* mul_w1) override {
        check_reps(reps);
        std::vector<VanillaGate<F>> gates(ng);
        for (size_t q = 0; q < ng; q++) {
            VanillaGate<F>& gt = gates[q];
            gt.has_const = has_const[q] != 0;
            gt.c = gt.has_const ? F::from_limbs(consts + q * F::LIMBS) : F::zero();
            for (uint64_t e = add_ptr[q]; e < add_ptr[q + 1]; e++) gt.adds.push_back({F::from_limbs(add_coef + e * F::LIMBS), (int)add_in[e], (size_t)add_wire[e]});
            for (uint64_t e = mul_ptr[q]; e < mul_ptr[q + 1]; e++)
                gt.muls.push_back({F::from_limbs(mul_coef + e * F::LIMBS), (int)mul_in0[e], (size_t)mul_w0[e], (int)mul_in1[e], (size_t)mul_w1[e]});
        }
        return g.c.insert(BfvEncrypt<F>::vanilla(arity, log2_sub, std::move(gates), reps));
    }
    void connect(int from, int to) override {
        if (from < 0 || to < 0 || from >= (int)g.c.nodes.size() || to >= (int)g.c.nodes.size()) throw OracleError("connect: no such node");
        g.c.connect(from, to);
    }
    void evaluate(const uint64_t* inputs) override {  // the input nodes' values back to back, insertion order
        std::vector<std::vector<F>> in;
        size_t off = 0;
        for (auto& n : g.c.nodes)
            if (n.kind == NODE_INPUT) { in.push_back(load_base<F>(inputs + off * F::LIMBS, n.out_len())); off += n.out_len(); }
        val = g.c.evaluate(in);
    }
    size_t value(int id, uint64_t* out) override {
        const auto& v = val.at(id);
        if (out) for (size_t i = 0; i < v.size(); i++) v[i].to_limbs(out + i * F::LIMBS);
        return v.size();
    }
    static std::vector<EvalClaim<F>> output_claims(size_t n, const size_t* lens, const uint64_t* pts, const uint64_t* vals) {
        std::vector<EvalClaim<F>> oc(n);
        size_t off = 0;
        for (size_t i = 0; i < n; i++) {
            for (size_t k = 0; k < lens[i]; k++) oc[i].point.push_back(load_ext<F, E>(pts + (off + k) * EL));
            off += lens[i];
            oc[i].value = load_ext<F, E>(vals + i * EL);
        }
        return oc;
    }
    size_t prove(size_t n, const size_t* lens, const uint64_t* pts, const uint64_t* vals, uint8_t* proof, size_t cap) override {
        if (val.size() != g.c.nodes.size()) throw OracleError("prove_gkr: evaluate the circuit first");
        Transcript<F> tr;
        claims = g.prove_gkr(val, output_claims(n, lens, pts, vals), tr);
        if (tr.stream.size() <= cap) memcpy(proof, tr.stream.data(), tr.stream.size());
        return tr.stream.size();
    }
    void verify(size_t n, const size_t* lens, const uint64_t* pts, const uint64_t* vals, const uint8_t* proof, size_t len) override {
        claims.clear();
        Transcript<F> tr(proof, len);
        auto ic = g.verify_gkr(output_claims(n, lens, pts, vals), tr);
        if (tr.rd_pos != len) throw OracleError("verify_gkr: trailing bytes in proof");
        claims = ic;
    }
    size_t num_inputs() const override { return claims.size(); }
    size_t num_claims(size_t input) const override { return input < claims.size() ? claims[input].size() : 0; }
    size_t claim(size_t input, size_t k, uint64_t* point, uint64_t* value) const override {
        const EvalClaim<F>& cl = claims.at(input).at(k);
        if (point) for (size_t i = 0; i < cl.point.size(); i++) store_ext<F, E>(cl.point[i], point + i * EL);
        if (value) store_ext<F, E>(cl.value, value);
        return cl.point.size();
    }
};
}  // namespace

#define GUARD(...) try { __VA_ARGS__ } catch (const std::exception& e) { g_err = e.what(); return 1; }

extern "C" {
const char* hgt_last_error() { return g_err.c_str(); }
void* hgt_new(int field) {
    if (field == 0) return (Session*)new SessionT<Gl>();
    if (field == 1) return (Session*)new SessionT<Fr>();
    g_err = "unknown field";
    return nullptr;
}
void hgt_free(void* h) { delete (Session*)h; }
int hgt_insert_input(void* h, int log2_size, int reps, int* out_id) { GUARD(*out_id = ((Session*)h)->insert_input(log2_size, reps); return 0;) }
int hgt_insert_fft(void* h, int log2_size, int inverse, int* out_id) { GUARD(*out_id = ((Session*)h)->insert_fft(log2_size, inverse != 0); return 0;) }
int hgt_insert_vanilla(void* h, int arity, int log2_sub, int reps, size_t ng, const uint8_t* has_const, const uint64_t* consts, const uint64_t* add_ptr,
                       const uint64_t* add_coef, const uint32_t* add_in, const uint64_t* add_wire, const uint64_t* mul_ptr, const uint64_t* mul_coef,
                       const uint32_t* mul_in0, const uint64_t* mul_w0, const uint32_t* mul_in1, const uint64_t* mul_w1, int* out_id) {
    GUARD(*out_id = ((Session*)h)->insert_vanilla(arity, log2_sub, reps, ng, has_const, consts, add_ptr, add_coef, add_in, add_wire, mul_ptr, mul_coef,
                                                  mul_in0, mul_w0, mul_in1, mul_w1);
          return 0;)
}
int hgt_connect(void* h, int from, int to) { GUARD(((Session*)h)->connect(from, to); return 0;) }
int hgt_evaluate(void* h, const uint64_t* inputs) { GUARD(((Session*)h)->evaluate(inputs); return 0;) }
int hgt_value(void* h, int id, uint64_t* out, size_t* len) { GUARD(*len = ((Session*)h)->value(id, out); return 0;) }
// prove_gkr from a fresh transcript; *len = proof size (the bytes are copied when they fit in cap)
int hgt_prove(void* h, size_t n, const size_t* lens, const uint64_t* pts, const uint64_t* vals, uint8_t* proof, size_t cap, size_t* len) {
    GUARD(*len = ((Session*)h)->prove(n, lens, pts, vals, proof, cap); return 0;)
}
int hgt_verify(void* h, size_t n, const size_t* lens, const uint64_t* pts, const uint64_t* vals, const uint8_t* proof, size_t len) {
    GUARD(((Session*)h)->verify(n, lens, pts, vals, proof, len); return 0;)
}
// the claims on the input nodes (insertion order) left by the last prove / verify
size_t hgt_num_inputs(void* h) { return ((Session*)h)->num_inputs(); }
size_t hgt_num_claims(void* h, size_t input) { return ((Session*)h)->num_claims(input); }
int hgt_claim(void* h, size_t input, size_t k, uint64_t* point, uint64_t* value, size_t* nvars) {
    GUARD(*nvars = ((Session*)h)->claim(input, k, point, value); return 0;)
}
}
