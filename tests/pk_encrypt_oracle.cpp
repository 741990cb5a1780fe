// TEST INFRASTRUCTURE ONLY (tests/test_pk_encrypt.py compiles it with g++ next to the oracle; the product never links it).
// An independent CPU restatement of the BFV public-key-encryption proof, for every modulus i < K over Z[x]:
//   ct0_i = pk0_i u + e0 + k0_i k1 + r1_i q_i + r2_i (x^n + 1)
//   ct1_i = pk1_i u + e1           + p1_i q_i + p2_i (x^n + 1)
// The circuit is written here from its node list (DESIGN.md section 3, assumption A12), not from the library's bfv_pk_configure, on
// the oracle's circuit, Lasso node and transcript (oracle/gkr.hpp), which prove every node shape it uses. C entries: build the
// circuit, evaluate (the Lasso node's input layer, sum0, sum1), prove (bytes and input claims) and verify, for both fields.
#include <cstring>
#include <string>

#include "gkr.hpp"

using namespace hgo;

namespace {
thread_local std::string g_err;

struct PkParams {
    int log2_size, K;
    std::vector<uint64_t> qis, k0is, r1, r2, p1, p2;
    uint64_t u_bound, e_bound, k1_bound;
};

template <class F> std::vector<F> load_base(const uint64_t* p, size_t n) {
    std::vector<F> v(n);
    for (size_t i = 0; i < n; i++) v[i] = F::from_limbs(p + i * F::LIMBS);
    return v;
}
template <class F, class E> void store_ext(const E& e, uint64_t* p) {
    F b[2]; e.as_bases(b);
    for (int i = 0; i < E::DEGREE; i++) b[i].to_limbs(p + i * F::LIMBS);
}

template <class F> struct BfvPkEncrypt {
    typedef typename ExtOf<F>::type E;
    typedef BfvEncrypt<F> B;  // node constructors
    typedef VanillaGate<F> G;
    PkParams P;
    Circuit<F> c;
    Preprocessing pp;
    int lasso_num_vars = 0, lasso_in = -1, sum0 = -1, sum1 = -1;

    explicit BfvPkEncrypt(const PkParams& params) : P(params) {
        const int L = P.log2_size, K = P.K, n_log2 = L - 1;
        const size_t N2 = (size_t)1 << L, n = N2 / 2;
        if (L < 2 || K < 1 || (K & (K - 1))) throw OracleError("BfvPkEncrypt: bad parameters");
        // preprocessing: [2U+1, 2E+1, 2K1+1] + 2 R1 + 1 + 2 P1 + 1 + 2 R2 + 1 + 2 P2 + 1 (equal ids collapse)
        std::vector<uint64_t> bounds = {P.u_bound * 2 + 1, P.e_bound * 2 + 1, P.k1_bound * 2 + 1};
        for (auto* v : {&P.r1, &P.p1, &P.r2, &P.p2}) for (int i = 0; i < K; i++) bounds.push_back((*v)[i] * 2 + 1);
        pp = Preprocessing::preprocess(bounds, 4, 16);
        // 1. inputs u, e0, e1, k1
        const int u = c.insert(B::input(L, 1)), e0 = c.insert(B::input(L, 1)), e1 = c.insert(B::input(L, 1)), k1 = c.insert(B::input(L, 1));
        // 2. e0s, e1s (K relays each), k1kis (k1 k0_i)
        std::vector<G> g;
        for (int i = 0; i < K; i++) for (size_t j = 0; j < N2; j++) g.push_back(G::relay(0, j));
        const int e0s = c.insert(B::vanilla(1, L, g, 1));
        const int e1s = c.insert(B::vanilla(1, L, g, 1));
        g.clear();
        for (int i = 0; i < K; i++) for (size_t j = 0; j < N2; j++) g.push_back(B::relay_mul_const(0, j, F::from_u64(P.k0is[i])));
        const int k1kis = c.insert(B::vanilla(1, L, g, 1));
        c.connect(e0, e0s); c.connect(e1, e1s); c.connect(k1, k1kis);
        // 3. pk0is, pk1is, r1is, p1is
        std::vector<int> pk0, pk1, r1, p1;
        for (auto* v : {&pk0, &pk1, &r1, &p1}) for (int i = 0; i < K; i++) v->push_back(c.insert(B::input(L, 1)));
        // 4. r1iqis, p1iqis
        g.clear();
        for (int i = 0; i < K; i++) for (size_t j = 0; j < N2; j++) g.push_back(B::relay_mul_const(i, j, F::from_u64(P.qis[i])));
        const int r1iqis = c.insert(B::vanilla(K, L, g, 1));
        const int p1iqis = c.insert(B::vanilla(K, L, g, 1));
        for (int x : r1) c.connect(x, r1iqis);
        for (int x : p1) c.connect(x, p1iqis);
        // 5. r2is, p2is: n x K each
        const int r2is = c.insert(B::input(n_log2, K)), p2is = c.insert(B::input(n_log2, K));
        // 6. chunks of 2n of each, the r2 ones first
        const size_t q2_len = n * K;
        const int q2_log2 = n_log2 + ilog2_u64(K);
        auto chunks = [&](int from) {
            std::vector<int> out;
            for (size_t start = 0; start < q2_len; start += N2) {
                std::vector<G> h;
                for (size_t j = start; j < std::min(start + N2, q2_len); j++) h.push_back(G::relay(0, j));
                h.resize(N2, G::constant(F::zero()));
                const int nd = c.insert(B::vanilla(1, q2_log2, h, 1));
                c.connect(from, nd);
                out.push_back(nd);
            }
            return out;
        };
        const std::vector<int> r2c = chunks(r2is), p2c = chunks(p2is);
        // 7. the Lasso node's input layer: r1is | p1is | r2 chunks | p2 chunks | u | e0 | e1 | k1, each element plus its own bound
        std::vector<int> ins;
        std::vector<std::vector<uint64_t>> shift;  // per input, per wire
        for (int i = 0; i < K; i++) { ins.push_back(r1[i]); shift.emplace_back(N2, P.r1[i]); }
        for (int i = 0; i < K; i++) { ins.push_back(p1[i]); shift.emplace_back(N2, P.p1[i]); }
        for (auto pr : {std::make_pair(&r2c, &P.r2), std::make_pair(&p2c, &P.p2)})
            for (size_t q = 0; q < pr.first->size(); q++) {
                ins.push_back((*pr.first)[q]);
                std::vector<uint64_t> s(N2);
                for (size_t j = 0; j < N2; j++) { size_t i = (q * N2 + j) / n; if (i >= (size_t)K) i = 0; s[j] = (*pr.second)[i]; }
                shift.push_back(s);
            }
        for (auto pr : {std::make_pair(u, P.u_bound), std::make_pair(e0, P.e_bound), std::make_pair(e1, P.e_bound), std::make_pair(k1, P.k1_bound)}) {
            ins.push_back(pr.first); shift.emplace_back(N2, pr.second);
        }
        g.clear();
        for (size_t t = 0; t < ins.size(); t++) for (size_t j = 0; j < N2; j++) g.push_back(B::relay_add_const((int)t, j, F::from_u64(shift[t][j])));
        lasso_in = c.insert(B::vanilla((int)ins.size(), L, g, 1));
        // 8. the Lasso node; lookup segments in the input layer's order
        std::vector<int> rows;
        auto push = [&](uint64_t b, size_t cnt) { const int li = pp.lookup_id_to_index.at(RangeLookup{b * 2 + 1}.id()); rows.insert(rows.end(), cnt, li); };
        const size_t seg2 = K == 1 ? N2 : n;
        for (int i = 0; i < K; i++) push(P.r1[i], N2);
        for (int i = 0; i < K; i++) push(P.p1[i], N2);
        for (int i = 0; i < K; i++) push(P.r2[i], seg2);
        for (int i = 0; i < K; i++) push(P.p2[i], seg2);
        push(P.u_bound, N2); push(P.e_bound, N2); push(P.e_bound, N2); push(P.k1_bound, N2);
        while (((size_t)1 << lasso_num_vars) < rows.size()) lasso_num_vars++;
        GkrNode<F> ln; ln.kind = NODE_LASSO; ln.lasso = std::make_shared<LassoNode<F>>(pp, lasso_num_vars, rows);
        const int lasso = c.insert(ln);
        for (int x : ins) c.connect(x, lasso_in);
        c.connect(lasso_in, lasso);
        // 9. u_eval = FFT(u), u_copy; per component a relay of arity K over IFFT(FFT(pk_i) . u_copy)
        const int u_eval = c.insert(B::fft(L, false));
        c.connect(u, u_eval);
        g.clear();
        for (size_t j = 0; j < N2; j++) g.push_back(G::relay(0, j));
        const int u_copy = c.insert(B::vanilla(1, L, g, 1));
        c.connect(u_eval, u_copy);
        auto products = [&](const std::vector<int>& pks) {
            std::vector<G> h;
            for (int i = 0; i < K; i++) for (size_t j = 0; j < N2; j++) h.push_back(G::relay(i, j));
            const int par = c.insert(B::vanilla(K, L, h, 1));
            h.clear();
            for (size_t j = 0; j < N2; j++) h.push_back(G::mul(0, j, 1, j));
            for (int i = 0; i < K; i++) {
                const int ev = c.insert(B::fft(L, false));
                const int m = c.insert(B::vanilla(2, L, h, 1));
                const int iv = c.insert(B::fft(L, true));
                c.connect(pks[i], ev);
                c.connect(u_copy, m); c.connect(ev, m);
                c.connect(m, iv);
                c.connect(iv, par);
            }
            return par;
        };
        const int pk0u = products(pk0), pk1u = products(pk1);
        // 10. q2_i (x^n + 1) for r2 and p2
        g.clear();
        for (int half = 0; half < 2; half++) {
            for (size_t j = 0; j + 1 < n; j++) g.push_back(G::relay(0, j));
            g.push_back(G::constant(F::zero()));
        }
        const int cyclo0 = c.insert(B::vanilla(1, n_log2, g, K));
        const int cyclo1 = c.insert(B::vanilla(1, n_log2, g, K));
        c.connect(r2is, cyclo0); c.connect(p2is, cyclo1);
        // 11. sum0 (arity 5), sum1 (arity 4), K reps each
        g.clear();
        for (size_t j = 0; j < N2; j++) g.push_back(G::sum({{0, j}, {1, j}, {2, j}, {3, j}, {4, j}}));
        sum0 = c.insert(B::vanilla(5, L, g, K));
        g.clear();
        for (size_t j = 0; j < N2; j++) g.push_back(G::sum({{0, j}, {1, j}, {2, j}, {3, j}}));
        sum1 = c.insert(B::vanilla(4, L, g, K));
        for (int x : {pk0u, e0s, k1kis, r1iqis, cyclo0}) c.connect(x, sum0);
        for (int x : {pk1u, e1s, p1iqis, cyclo1}) c.connect(x, sum1);
    }
    int ct_log2() const { return P.log2_size + ilog2_u64(P.K); }

    std::vector<EvalClaim<F>> output_claims(Transcript<F>& tr, const std::vector<F>& ct0, const std::vector<F>& ct1) const {
        std::vector<E> pt0 = tr.squeeze_n(ct_log2());
        const E v0 = mle_evaluate<E, F>(ct0, pt0);
        std::vector<E> pt1 = tr.squeeze_n(ct_log2());
        const E v1 = mle_evaluate<E, F>(ct1, pt1);
        return {{{}, E::zero()}, {pt0, v0}, {pt1, v1}};
    }
};

struct Session {
    virtual ~Session() {}
    virtual void evaluate(const uint64_t* inputs) = 0;
    virtual size_t value(int which, uint64_t* out) = 0;
    virtual size_t prove(const uint64_t* ct0, const uint64_t* ct1, uint8_t* proof, size_t cap) = 0;
    virtual void verify(const uint64_t* inputs, const uint64_t* ct0, const uint64_t* ct1, const uint8_t* proof, size_t len) = 0;
    virtual int lasso_num_vars() const = 0;
    virtual size_t num_inputs() const = 0;
    virtual size_t num_claims(size_t input) const = 0;
    virtual size_t claim(size_t input, size_t k, uint64_t* point, uint64_t* value) const = 0;
};
template <class F> struct SessionT : Session {
    typedef typename ExtOf<F>::type E;
    static constexpr size_t EL = E::DEGREE * F::LIMBS;
    BfvPkEncrypt<F> b;
    std::vector<std::vector<F>> val;
    std::vector<std::vector<EvalClaim<F>>> claims;
    explicit SessionT(const PkParams& P) : b(P) {}
    size_t ct_len() const { return (size_t)1 << b.ct_log2(); }
    std::vector<std::vector<F>> load_inputs(const uint64_t* inputs) const {  // the input nodes' values back to back, insertion order
        std::vector<std::vector<F>> in;
        size_t off = 0;
        for (auto& n : b.c.nodes)
            if (n.kind == NODE_INPUT) { in.push_back(load_base<F>(inputs + off * F::LIMBS, n.out_len())); off += n.out_len(); }
        return in;
    }
    void evaluate(const uint64_t* inputs) override { val = b.c.evaluate(load_inputs(inputs)); }
    size_t value(int which, uint64_t* out) override {
        const int id = which == 0 ? b.lasso_in : which == 1 ? b.sum0 : b.sum1;
        const auto& v = val.at(id);
        if (out) for (size_t i = 0; i < v.size(); i++) v[i].to_limbs(out + i * F::LIMBS);
        return v.size();
    }
    size_t prove(const uint64_t* ct0, const uint64_t* ct1, uint8_t* proof, size_t cap) override {
        if (val.size() != b.c.nodes.size()) throw OracleError("prove: evaluate the circuit first");
        Transcript<F> tr;
        const auto oc = b.output_claims(tr, load_base<F>(ct0, ct_len()), load_base<F>(ct1, ct_len()));
        claims = b.c.prove_gkr(val, oc, tr);
        if (tr.stream.size() <= cap) memcpy(proof, tr.stream.data(), tr.stream.size());
        return tr.stream.size();
    }
    void verify(const uint64_t* inputs, const uint64_t* ct0, const uint64_t* ct1, const uint8_t* proof, size_t len) override {
        claims.clear();
        Transcript<F> tr(proof, len);
        const auto oc = b.output_claims(tr, load_base<F>(ct0, ct_len()), load_base<F>(ct1, ct_len()));
        auto ic = b.c.verify_gkr(oc, tr);
        if (tr.rd_pos != len) throw OracleError("verify: trailing bytes in proof");
        const auto in = load_inputs(inputs);
        if (ic.size() != in.size()) throw OracleError("verify: input count mismatch");
        for (size_t i = 0; i < in.size(); i++)
            for (auto& cl : ic[i])
                if (mle_evaluate<E, F>(in[i], cl.point) != cl.value) throw OracleError("verify: input claim does not match the input");
        claims = ic;
    }
    int lasso_num_vars() const override { return b.lasso_num_vars; }
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
const char* hgpk_last_error() { return g_err.c_str(); }
// bounds6: K entries each of qis, k0is, R1, R2, P1, P2, back to back
int hgpk_new(int field, int log2_size, int K, const uint64_t* bounds6, uint64_t u_bound, uint64_t e_bound, uint64_t k1_bound, void** out) {
    GUARD(
        PkParams P;
        P.log2_size = log2_size; P.K = K; P.u_bound = u_bound; P.e_bound = e_bound; P.k1_bound = k1_bound;
        for (auto* v : {&P.qis, &P.k0is, &P.r1, &P.r2, &P.p1, &P.p2}) { v->assign(bounds6, bounds6 + K); bounds6 += K; }
        if (field == 0) *out = (Session*)new SessionT<Gl>(P);
        else if (field == 1) *out = (Session*)new SessionT<Fr>(P);
        else throw OracleError("unknown field");
        return 0;)
}
void hgpk_free(void* h) { delete (Session*)h; }
// the A3 / A3' / A5 switches (oracle/protocol.hpp: Assumptions) of this restatement; ids as hg_ctx_set_option
void hgpk_set_assumption(int which, int value) {
    if (which == 3) assumptions().a3_wire = value;
    if (which == 31) assumptions().a3_h1 = value;
    if (which == 5) assumptions().a5_ascending = value;
}
int hgpk_lasso_num_vars(void* h) { return ((Session*)h)->lasso_num_vars(); }
int hgpk_evaluate(void* h, const uint64_t* inputs) { GUARD(((Session*)h)->evaluate(inputs); return 0;) }
// which: 0 the Lasso node's input layer, 1 sum0, 2 sum1
int hgpk_value(void* h, int which, uint64_t* out, size_t* len) { GUARD(*len = ((Session*)h)->value(which, out); return 0;) }
// the proof of the last evaluation from a fresh transcript; *len = proof size (the bytes are copied when they fit in cap)
int hgpk_prove(void* h, const uint64_t* ct0, const uint64_t* ct1, uint8_t* proof, size_t cap, size_t* len) {
    GUARD(*len = ((Session*)h)->prove(ct0, ct1, proof, cap); return 0;)
}
int hgpk_verify(void* h, const uint64_t* inputs, const uint64_t* ct0, const uint64_t* ct1, const uint8_t* proof, size_t len) {
    GUARD(((Session*)h)->verify(inputs, ct0, ct1, proof, len); return 0;)
}
size_t hgpk_num_inputs(void* h) { return ((Session*)h)->num_inputs(); }
size_t hgpk_num_claims(void* h, size_t input) { return ((Session*)h)->num_claims(input); }
int hgpk_claim(void* h, size_t input, size_t k, uint64_t* point, uint64_t* value, size_t* nvars) {
    GUARD(*nvars = ((Session*)h)->claim(input, k, point, value); return 0;)
}
}
