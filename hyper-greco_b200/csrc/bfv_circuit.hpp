// BfvEncryptBlock::configure (/root/reference/bfv-gkr/src/sk_encryption_circuit.rs:86-293) in the host library: the circuit topology
// of the BFV secret-key-encryption proof, node for node and connection for connection, built through the same insert / connect
// calls the C ABI exposes (hg_circuit_insert_* / hg_circuit_connect). A Rust caller that keeps `configure` as it is binds those
// calls one by one; a caller that only wants the finished circuit (bench, tests, the verifier) calls hg_bfv_configure.
// Works on any circuit type with insert_input / insert_fft / insert_vanilla(VanillaDesc) / connect: the device circuit
// (GkrCircuitDev) and the host-only description (GkrVerifierHost).
#pragma once
#include <functional>

#include "gkr_dev.cuh"

namespace hg {

struct BfvCircuitParams {  // BfvSkEncryptConstans (constants/mod.rs:16-35) for K moduli; L = N_LOG2 + 1 (:81-83)
    size_t log2_size = 0, K = 0;
    std::vector<uint64_t> qis, k0is, r1_bounds, r2_bounds;
    uint64_t s_bound = 0, e_bound = 0, k1_bound = 0;
};
struct BfvCircuitIds { int s = -1, e = -1, k1 = -1, lasso_in = -1, lasso = -1, sum = -1; };

// gates `const + sum coef * input[in][wire]`, one additive edge per gate unless add_ptr is given
template <int LIMBS> struct VanillaBuilder {
    VanillaDesc d;
    VanillaBuilder(size_t arity, size_t log2_sub, size_t reps) { d.arity = arity; d.log2_sub = log2_sub; d.num_reps = reps; d.add_ptr.push_back(0); d.mul_ptr.push_back(0); }
    void felt(std::vector<uint64_t>& v, uint64_t x) { v.push_back(x); for (int l = 1; l < LIMBS; l++) v.push_back(0); }
    // relay_mul_const / relay_add_const / relay / constant (:525-531 and VanillaGate::{relay, constant})
    void gate(bool has_const, uint64_t c, const std::vector<std::tuple<uint64_t, uint32_t, uint64_t>>& adds) {
        d.has_const.push_back(has_const ? 1 : 0);
        felt(d.consts, c);
        for (auto& a : adds) { felt(d.add_coef, std::get<0>(a)); d.add_in.push_back(std::get<1>(a)); d.add_wire.push_back(std::get<2>(a)); }
        d.add_ptr.push_back(d.add_in.size());
        d.mul_ptr.push_back(d.mul_in0.size());
        d.n_gates++;
    }
    void mul_gate(uint32_t i0, uint64_t w0, uint32_t i1, uint64_t w1) {  // VanillaGate::mul((i0, w0), (i1, w1))
        d.has_const.push_back(0);
        felt(d.consts, 0);
        felt(d.mul_coef, 1); d.mul_in0.push_back(i0); d.mul_w0.push_back(w0); d.mul_in1.push_back(i1); d.mul_w1.push_back(w1);
        d.add_ptr.push_back(d.add_in.size());
        d.mul_ptr.push_back(d.mul_in0.size());
        d.n_gates++;
    }
};

// insert_lasso() inserts the Lasso node (device node or host description) and returns its id
template <int LIMBS, class Ckt> BfvCircuitIds bfv_configure(Ckt& c, const BfvCircuitParams& P, const std::function<int()>& insert_lasso) {
    typedef VanillaBuilder<LIMBS> VB;
    const size_t L = P.log2_size, K = P.K, N2 = (size_t)1 << L;
    if (L < 2 || K < 1 || P.qis.size() < K || P.k0is.size() < K || P.r1_bounds.size() < K || P.r2_bounds.size() < K) throw std::runtime_error("bfv_configure: bad parameters");
    size_t log2K = 0;
    while (((size_t)1 << log2K) < K) log2K++;
    if (((size_t)1 << log2K) != K) throw std::runtime_error("bfv_configure: K must be a power of two (ct0is_log2_size, sk_encryption_circuit.rs:519-522)");
    BfvCircuitIds id;
    id.s = c.insert_input(L, 1); id.e = c.insert_input(L, 1); id.k1 = c.insert_input(L, 1);
    int es, k1kis;
    {   // es: K copies of e (:97-103); k1kis: k1 * k0_i (:105-115)
        VB a(1, L, 1), b(1, L, 1);
        for (size_t i = 0; i < K; i++)
            for (size_t j = 0; j < N2; j++) { a.gate(false, 0, {{1, 0, j}}); b.gate(false, 0, {{P.k0is[i], 0, j}}); }
        es = c.insert_vanilla(a.d);
        k1kis = c.insert_vanilla(b.d);
    }
    c.connect(id.e, es);
    c.connect(id.k1, k1kis);
    std::vector<int> ais, r1is;
    for (size_t i = 0; i < K; i++) ais.push_back(c.insert_input(L, 1));
    for (size_t i = 0; i < K; i++) r1is.push_back(c.insert_input(L, 1));
    int r1iqis;
    {   // r1i * q_i (:130-141)
        VB a(K, L, 1);
        for (size_t i = 0; i < K; i++) for (size_t j = 0; j < N2; j++) a.gate(false, 0, {{P.qis[i], (uint32_t)i, j}});
        r1iqis = c.insert_vanilla(a.d);
    }
    for (int r : r1is) c.connect(r, r1iqis);
    const size_t n_log2 = L - 1;
    const int r2is = c.insert_input(n_log2, K);                               // :147
    const size_t r2_log2 = n_log2 + log2K;
    std::vector<int> chunks;
    for (size_t start = 0; start < ((size_t)1 << r2_log2); start += N2) {     // :150-161
        const size_t cnt = std::min(N2, ((size_t)1 << r2_log2) - start);
        VB a(1, r2_log2, 1);
        for (size_t j = 0; j < N2; j++) {
            if (j < cnt) a.gate(false, 0, {{1, 0, start + j}});
            else a.gate(true, 0, {});
        }
        const int nd = c.insert_vanilla(a.d);
        c.connect(r2is, nd);
        chunks.push_back(nd);
    }
    {   // lasso_inputs_batched: every range-checked vector shifted by its bound (:163-181; Q7: every r2 chunk by R2_BOUNDS[0])
        std::vector<uint64_t> shifts(P.r1_bounds.begin(), P.r1_bounds.begin() + K);
        for (size_t q = 0; q < chunks.size(); q++) shifts.push_back(P.r2_bounds[0]);
        shifts.push_back(P.s_bound); shifts.push_back(P.e_bound); shifts.push_back(P.k1_bound);
        VB a(shifts.size(), L, 1);
        for (size_t i = 0; i < shifts.size(); i++) for (size_t j = 0; j < N2; j++) a.gate(true, shifts[i], {{1, (uint32_t)i, j}});
        id.lasso_in = c.insert_vanilla(a.d);
    }
    id.lasso = insert_lasso();                                                // :205-209
    for (int r : r1is) c.connect(r, id.lasso_in);
    for (int ch : chunks) c.connect(ch, id.lasso_in);
    c.connect(id.s, id.lasso_in); c.connect(id.e, id.lasso_in); c.connect(id.k1, id.lasso_in);
    c.connect(id.lasso_in, id.lasso);
    const int s_eval = c.insert_fft(L, false);                                // :224
    c.connect(id.s, s_eval);
    int s_copy, sai_par;
    {
        VB a(1, L, 1);                                                        // :227-235
        for (size_t j = 0; j < N2; j++) a.gate(false, 0, {{1, 0, j}});
        s_copy = c.insert_vanilla(a.d);
        VB b(K, L, 1);                                                        // :237-243
        for (size_t i = 0; i < K; i++) for (size_t j = 0; j < N2; j++) b.gate(false, 0, {{1, (uint32_t)i, j}});
        c.connect(s_eval, s_copy);
        sai_par = c.insert_vanilla(b.d);
    }
    for (int ai : ais) {                                                      // :245-260
        const int ai_eval = c.insert_fft(L, false);
        VB m(2, L, 1);
        for (size_t j = 0; j < N2; j++) m.mul_gate(0, j, 1, j);
        const int sai_eval = c.insert_vanilla(m.d);
        const int sai = c.insert_fft(L, true);
        c.connect(ai, ai_eval);
        c.connect(s_copy, sai_eval);
        c.connect(ai_eval, sai_eval);
        c.connect(sai_eval, sai);
        c.connect(sai, sai_par);
    }
    int cyclo;
    {   // r2i * (x^n + 1): the n-1 coefficients of r2i twice, each run followed by a zero (:262-278)
        const size_t n = (size_t)1 << n_log2;
        VB a(1, n_log2, K);
        for (int half = 0; half < 2; half++) {
            for (size_t j = 0; j + 1 < n; j++) a.gate(false, 0, {{1, 0, j}});
            a.gate(true, 0, {});
        }
        cyclo = c.insert_vanilla(a.d);
    }
    {   // sum of the five parts (:280-285)
        VB a(5, L, K);
        for (size_t j = 0; j < N2; j++) a.gate(false, 0, {{1, 0, j}, {1, 1, j}, {1, 2, j}, {1, 3, j}, {1, 4, j}});
        id.sum = c.insert_vanilla(a.d);
    }
    c.connect(r2is, cyclo);
    c.connect(sai_par, id.sum); c.connect(es, id.sum); c.connect(k1kis, id.sum); c.connect(r1iqis, id.sum); c.connect(cyclo, id.sum);
    return id;
}

// ---- BFV public-key encryption (Greco's second relation), for every modulus i < K over Z[x]:
//   ct0_i = pk0_i u + e0 + k0_i k1 + r1_i q_i + r2_i (x^n + 1)
//   ct1_i = pk1_i u + e1           + p1_i q_i + p2_i (x^n + 1)
// The topology has no reference implementation: it is the SK circuit's, doubled where the relation doubles (DESIGN.md section 3,
// assumption A12). Node insertion order fixes the input order, the output order and the proof bytes.
struct BfvPkCircuitParams {
    size_t log2_size = 0, K = 0;
    std::vector<uint64_t> qis, k0is, r1_bounds, r2_bounds, p1_bounds, p2_bounds;
    uint64_t u_bound = 0, e_bound = 0, k1_bound = 0;
};
struct BfvPkCircuitIds { int u = -1, e0 = -1, e1 = -1, k1 = -1, lasso_in = -1, lasso = -1, sum0 = -1, sum1 = -1; };

template <int LIMBS, class Ckt> BfvPkCircuitIds bfv_pk_configure(Ckt& c, const BfvPkCircuitParams& P, const std::function<int()>& insert_lasso) {
    typedef VanillaBuilder<LIMBS> VB;
    const size_t L = P.log2_size, K = P.K, N2 = (size_t)1 << L;
    if (L < 2 || K < 1 || P.qis.size() < K || P.k0is.size() < K || P.r1_bounds.size() < K || P.r2_bounds.size() < K || P.p1_bounds.size() < K ||
        P.p2_bounds.size() < K)
        throw std::runtime_error("bfv_pk_configure: bad parameters");
    size_t log2K = 0;
    while (((size_t)1 << log2K) < K) log2K++;
    if (((size_t)1 << log2K) != K) throw std::runtime_error("bfv_pk_configure: K must be a power of two (the outputs are K blocks of 2n)");
    BfvPkCircuitIds id;
    id.u = c.insert_input(L, 1); id.e0 = c.insert_input(L, 1); id.e1 = c.insert_input(L, 1); id.k1 = c.insert_input(L, 1);
    int e0s, e1s, k1kis;
    {   // e0s, e1s: K copies of e0 / e1; k1kis: k1 * k0_i
        VB a(1, L, 1), b(1, L, 1), d(1, L, 1);
        for (size_t i = 0; i < K; i++)
            for (size_t j = 0; j < N2; j++) { a.gate(false, 0, {{1, 0, j}}); b.gate(false, 0, {{1, 0, j}}); d.gate(false, 0, {{P.k0is[i], 0, j}}); }
        e0s = c.insert_vanilla(a.d);
        e1s = c.insert_vanilla(b.d);
        k1kis = c.insert_vanilla(d.d);
    }
    c.connect(id.e0, e0s);
    c.connect(id.e1, e1s);
    c.connect(id.k1, k1kis);
    std::vector<int> pk0is, pk1is, r1is, p1is;
    for (size_t i = 0; i < K; i++) pk0is.push_back(c.insert_input(L, 1));
    for (size_t i = 0; i < K; i++) pk1is.push_back(c.insert_input(L, 1));
    for (size_t i = 0; i < K; i++) r1is.push_back(c.insert_input(L, 1));
    for (size_t i = 0; i < K; i++) p1is.push_back(c.insert_input(L, 1));
    int r1iqis, p1iqis;
    {   // r1_i * q_i, p1_i * q_i
        VB a(K, L, 1), b(K, L, 1);
        for (size_t i = 0; i < K; i++) for (size_t j = 0; j < N2; j++) { a.gate(false, 0, {{P.qis[i], (uint32_t)i, j}}); b.gate(false, 0, {{P.qis[i], (uint32_t)i, j}}); }
        r1iqis = c.insert_vanilla(a.d);
        p1iqis = c.insert_vanilla(b.d);
    }
    for (int r : r1is) c.connect(r, r1iqis);
    for (int p : p1is) c.connect(p, p1iqis);
    const size_t n_log2 = L - 1, n = (size_t)1 << n_log2;
    const int r2is = c.insert_input(n_log2, K), p2is = c.insert_input(n_log2, K);
    const size_t q2_log2 = n_log2 + log2K;
    // chunks of 2n of a quotient vector (K blocks of n), the SK circuit's chunking; for K = 1 the second half is zero padding
    auto chunk = [&](int from, std::vector<int>& out) {
        for (size_t start = 0; start < ((size_t)1 << q2_log2); start += N2) {
            const size_t cnt = std::min(N2, ((size_t)1 << q2_log2) - start);
            VB a(1, q2_log2, 1);
            for (size_t j = 0; j < N2; j++) {
                if (j < cnt) a.gate(false, 0, {{1, 0, start + j}});
                else a.gate(true, 0, {});
            }
            const int nd = c.insert_vanilla(a.d);
            c.connect(from, nd);
            out.push_back(nd);
        }
    };
    std::vector<int> r2_chunks, p2_chunks;
    chunk(r2is, r2_chunks);
    chunk(p2is, p2_chunks);
    {   // every range-checked element shifted by its own vector's bound: r1is | p1is | r2 chunks | p2 chunks | u | e0 | e1 | k1. A chunk
        // element at flat index f belongs to modulus f / n (modulus 0 for the zero padding of K = 1)
        const size_t arity = 2 * K + r2_chunks.size() + p2_chunks.size() + 4;
        VB a(arity, L, 1);
        uint32_t in = 0;
        auto whole = [&](uint64_t shift) { for (size_t j = 0; j < N2; j++) a.gate(true, shift, {{1, in, j}}); in++; };
        auto chunks = [&](const std::vector<int>& ch, const std::vector<uint64_t>& bounds) {
            for (size_t q = 0; q < ch.size(); q++, in++)
                for (size_t j = 0; j < N2; j++) a.gate(true, bounds[std::min((q * N2 + j) / n, K - 1)], {{1, in, j}});
        };
        for (size_t i = 0; i < K; i++) whole(P.r1_bounds[i]);
        for (size_t i = 0; i < K; i++) whole(P.p1_bounds[i]);
        chunks(r2_chunks, P.r2_bounds);
        chunks(p2_chunks, P.p2_bounds);
        whole(P.u_bound); whole(P.e_bound); whole(P.e_bound); whole(P.k1_bound);
        id.lasso_in = c.insert_vanilla(a.d);
    }
    id.lasso = insert_lasso();
    for (int r : r1is) c.connect(r, id.lasso_in);
    for (int p : p1is) c.connect(p, id.lasso_in);
    for (int ch : r2_chunks) c.connect(ch, id.lasso_in);
    for (int ch : p2_chunks) c.connect(ch, id.lasso_in);
    c.connect(id.u, id.lasso_in); c.connect(id.e0, id.lasso_in); c.connect(id.e1, id.lasso_in); c.connect(id.k1, id.lasso_in);
    c.connect(id.lasso_in, id.lasso);
    const int u_eval = c.insert_fft(L, false);
    c.connect(id.u, u_eval);
    int u_copy;
    {   // one claim on FFT(u), as s_copy gives the SK circuit
        VB a(1, L, 1);
        for (size_t j = 0; j < N2; j++) a.gate(false, 0, {{1, 0, j}});
        u_copy = c.insert_vanilla(a.d);
        c.connect(u_eval, u_copy);
    }
    // a relay of arity K over the products pk_i * u = IFFT(FFT(pk_i) . u_copy)
    auto products = [&](const std::vector<int>& pks) {
        VB b(K, L, 1);
        for (size_t i = 0; i < K; i++) for (size_t j = 0; j < N2; j++) b.gate(false, 0, {{1, (uint32_t)i, j}});
        const int par = c.insert_vanilla(b.d);
        for (int pk : pks) {
            const int pk_eval = c.insert_fft(L, false);
            VB m(2, L, 1);
            for (size_t j = 0; j < N2; j++) m.mul_gate(0, j, 1, j);
            const int pku_eval = c.insert_vanilla(m.d);
            const int pku = c.insert_fft(L, true);
            c.connect(pk, pk_eval);
            c.connect(u_copy, pku_eval);
            c.connect(pk_eval, pku_eval);
            c.connect(pku_eval, pku);
            c.connect(pku, par);
        }
        return par;
    };
    const int pk0u_par = products(pk0is);
    const int pk1u_par = products(pk1is);
    auto cyclo = [&]() {  // q2_i * (x^n + 1): the n-1 coefficients of q2_i twice, each run followed by a zero
        VB a(1, n_log2, K);
        for (int half = 0; half < 2; half++) {
            for (size_t j = 0; j + 1 < n; j++) a.gate(false, 0, {{1, 0, j}});
            a.gate(true, 0, {});
        }
        return c.insert_vanilla(a.d);
    };
    const int cyclo0 = cyclo(), cyclo1 = cyclo();
    c.connect(r2is, cyclo0);
    c.connect(p2is, cyclo1);
    {
        VB a(5, L, K), b(4, L, K);
        for (size_t j = 0; j < N2; j++) {
            a.gate(false, 0, {{1, 0, j}, {1, 1, j}, {1, 2, j}, {1, 3, j}, {1, 4, j}});
            b.gate(false, 0, {{1, 0, j}, {1, 1, j}, {1, 2, j}, {1, 3, j}});
        }
        id.sum0 = c.insert_vanilla(a.d);
        id.sum1 = c.insert_vanilla(b.d);
    }
    c.connect(pk0u_par, id.sum0); c.connect(e0s, id.sum0); c.connect(k1kis, id.sum0); c.connect(r1iqis, id.sum0); c.connect(cyclo0, id.sum0);
    c.connect(pk1u_par, id.sum1); c.connect(e1s, id.sum1); c.connect(p1iqis, id.sum1); c.connect(cyclo1, id.sum1);
    return id;
}

}  // namespace hg
