// ORACLE — TEST INFRASTRUCTURE ONLY. Restatement of the GKR engine the reference takes from the un-vendored `gkr` crate
// (git https://github.com/han0110/gkr patched to https://github.com/nulltea/gkr-lasso, no rev; /root/reference/Cargo.toml:10,63-64)
// for exactly the node shapes bfv-gkr builds (sk_encryption_circuit.rs:86-293). PARITY UNPINNED: the crate's source is absent,
// so this follows the PUBLISHED algorithms (Libra-style layer sumcheck for linear layers, the zkCNN FFT-matrix sumcheck,
// an eq-weighted product sumcheck for the element-wise multiplication layer) and is anchored on what the reference's own
// tests pin: prove -> verify accepts, and every returned input claim equals the input's MLE at the claim point
// (sk_encryption_circuit.rs:512-516). Protocol per node (assumption A7/A8, documented in DESIGN.md section 3):
//     [T > 1 claims: squeeze alpha, weights alpha^t]  ->  sumcheck rounds (A3 wire format)  ->  write the input evaluations
#pragma once
#include <tuple>

#include "protocol.hpp"

namespace hgo {

template <class F> struct VanillaGate {  // VanillaGate::new(Option<F>, Vec<(Option<F>, (input, wire))>, Vec<(Option<F>, wire, wire)>)
    bool has_const = false;
    F c;
    std::vector<std::tuple<F, int, size_t>> adds;                       // coefficient (None = 1), (input index, wire)
    std::vector<std::tuple<F, int, size_t, int, size_t>> muls;          // coefficient, (input, wire), (input, wire)
    static VanillaGate relay(int in, size_t w) { VanillaGate g; g.adds.push_back({F::one(), in, w}); return g; }
    static VanillaGate constant(F c) { VanillaGate g; g.has_const = true; g.c = c; return g; }
    static VanillaGate mul(int i0, size_t w0, int i1, size_t w1) { VanillaGate g; g.muls.push_back({F::one(), i0, w0, i1, w1}); return g; }
    static VanillaGate sum(const std::vector<std::pair<int, size_t>>& ws) { VanillaGate g; for (auto& w : ws) g.adds.push_back({F::one(), w.first, w.second}); return g; }
};

enum NodeKind { NODE_INPUT, NODE_VANILLA, NODE_FFT, NODE_LASSO };

template <class F> struct EvalClaim {
    typedef typename ExtOf<F>::type E;
    std::vector<E> point;
    E value;
};

template <class F> struct GkrNode {
    typedef typename ExtOf<F>::type E;
    NodeKind kind = NODE_INPUT;
    int log2_size = 0, num_reps = 1;             // InputNode::new(log2_size, num_reps)
    // vanilla: VanillaNode::new(input_arity, log2_sub_input_size, gates, num_reps)
    int arity = 0, log2_sub_input = 0;
    std::vector<VanillaGate<F>> gates;
    bool fft_inverse = false;                    // FftNode::forward / ::inverse (log2_size)
    std::shared_ptr<LassoNode<F>> lasso;
    std::vector<int> preds, succs;

    size_t out_len() const {
        if (kind == NODE_INPUT) return (size_t)num_reps << log2_size;
        if (kind == NODE_FFT) return (size_t)1 << log2_size;
        if (kind == NODE_LASSO) return 1;
        size_t n = gates.size() * num_reps, p = 1;
        while (p < n) p <<= 1;
        return p;
    }
    // the only multiplicative layer of the circuit: out[i] = in0[i] * in1[i] (:246-250), one gate per input wire and num_reps 1. With
    // fewer gates than wires the product sumcheck would prove a sum that misses the unread wires, at a point shorter than the inputs'.
    bool elementwise_mul() const {
        if (kind != NODE_VANILLA || arity != 2 || num_reps != 1 || gates.size() != ((size_t)1 << log2_sub_input)) return false;
        for (size_t i = 0; i < gates.size(); i++) {
            auto& g = gates[i];
            if (g.has_const || !g.adds.empty() || g.muls.size() != 1) return false;
            auto& m = g.muls[0];
            if (std::get<0>(m) != F::one() || std::get<1>(m) != 0 || std::get<3>(m) != 1 || std::get<2>(m) != i || std::get<4>(m) != i) return false;
        }
        return true;
    }
    bool linear() const { for (auto& g : gates) if (!g.muls.empty()) return false; return kind == NODE_VANILLA; }
};

template <class F> struct Circuit {
    typedef typename ExtOf<F>::type E;
    std::vector<GkrNode<F>> nodes;
    int insert(const GkrNode<F>& n) { nodes.push_back(n); return (int)nodes.size() - 1; }
    void connect(int from, int to) { nodes[to].preds.push_back(from); nodes[from].succs.push_back(to); }

    // topological order (assumption A7): Kahn's algorithm, always taking the ready node with the smallest insertion index.
    // Insertion order itself is NOT topological (sai_par is inserted before the nodes that feed it, :237-260).
    std::vector<int> topo_order() const {
        std::vector<int> indeg(nodes.size()), order;
        for (size_t i = 0; i < nodes.size(); i++) indeg[i] = (int)nodes[i].preds.size();
        std::vector<char> done(nodes.size(), 0);
        for (size_t step = 0; step < nodes.size(); step++) {
            int pick = -1;
            for (size_t i = 0; i < nodes.size(); i++) if (!done[i] && indeg[i] == 0) { pick = (int)i; break; }
            if (pick < 0) throw OracleError("circuit has a cycle");
            done[pick] = 1;
            order.push_back(pick);
            for (int s : nodes[pick].succs) indeg[s]--;
        }
        return order;
    }

    // ---- Circuit::evaluate: values of every node, inputs given for the input nodes in insertion order
    std::vector<std::vector<F>> evaluate(const std::vector<std::vector<F>>& inputs) const {
        std::vector<std::vector<F>> val(nodes.size());
        {
            size_t next_in = 0;
            for (size_t id = 0; id < nodes.size(); id++)
                if (nodes[id].kind == NODE_INPUT) { val[id] = inputs.at(next_in++); if (val[id].size() != nodes[id].out_len()) throw OracleError("input size mismatch"); }
        }
        for (int id : topo_order()) {
            const auto& nd = nodes[id];
            if (nd.kind == NODE_INPUT) continue;
            if (nd.kind == NODE_LASSO) { val[id] = {F::zero()}; continue; }  // lasso.rs:53-55
            if (nd.kind == NODE_FFT) { val[id] = val[nd.preds.at(0)]; ntt_naive_order(val[id], nd.fft_inverse); continue; }
            std::vector<F> out(nd.out_len(), F::zero());
            const size_t ng = nd.gates.size(), sub = (size_t)1 << nd.log2_sub_input;
            for (int r = 0; r < nd.num_reps; r++)
                for (size_t g = 0; g < ng; g++) {
                    const auto& gt = nd.gates[g];
                    F v = gt.has_const ? gt.c : F::zero();
                    for (auto& a : gt.adds) v += std::get<0>(a) * val[nd.preds.at(std::get<1>(a))].at(r * sub + std::get<2>(a));
                    for (auto& m : gt.muls)
                        v += std::get<0>(m) * val[nd.preds.at(std::get<1>(m))].at(r * sub + std::get<2>(m)) * val[nd.preds.at(std::get<3>(m))].at(r * sub + std::get<4>(m));
                    out[r * ng + g] = v;
                }
            val[id].swap(out);
        }
        return val;
    }

    // ---- weights of the layer sumcheck: A[x] such that  sum_t alpha^t O~(z_t) = const + sum_x A[x] * X[x]
    // X = concatenation of the node's inputs, each padded to n_in = num_reps * 2^log2_sub_input, arity padded to a power of two
    static std::vector<E> combined_eq(const std::vector<EvalClaim<F>>& claims, E alpha, size_t out_len) {
        std::vector<E> w(out_len, E::zero());
        E p = E::one();
        for (auto& c : claims) {
            std::vector<E> eq = eq_xy(c.point);
            if (eq.size() != out_len) throw OracleError("claim point does not match the node's output size");
            for (size_t i = 0; i < out_len; i++) w[i] += p * eq[i];
            p *= alpha;
        }
        return w;
    }
    static size_t pad2(size_t n) { size_t p = 1; while (p < n) p <<= 1; return p; }

    struct Reduction { std::vector<E> A; std::vector<F> X; E constant; size_t n_in, a_pad; };
    Reduction linear_reduction(const GkrNode<F>& nd, const std::vector<E>& w, const std::vector<std::vector<F>>* val) const {
        Reduction R;
        R.n_in = (size_t)nd.num_reps << nd.log2_sub_input;
        R.a_pad = pad2(nd.arity);
        R.A.assign(R.a_pad * R.n_in, E::zero());
        R.constant = E::zero();
        const size_t ng = nd.gates.size(), sub = (size_t)1 << nd.log2_sub_input;
        for (int r = 0; r < nd.num_reps; r++)
            for (size_t g = 0; g < ng; g++) {
                const auto& gt = nd.gates[g];
                const E wg = w[r * ng + g];
                if (gt.has_const) R.constant += wg * gt.c;
                for (auto& a : gt.adds) R.A[std::get<1>(a) * R.n_in + r * sub + std::get<2>(a)] += wg * std::get<0>(a);
            }
        if (val) {
            R.X.assign(R.a_pad * R.n_in, F::zero());
            for (int k = 0; k < nd.arity; k++) std::copy((*val)[nd.preds[k]].begin(), (*val)[nd.preds[k]].end(), R.X.begin() + k * R.n_in);
        }
        return R;
    }
    // FFT-matrix weights (zkCNN): O = M I  =>  A[j] = sum_k w[k] M[k][j]; M symmetric, so A = transform(w)
    static std::vector<E> fft_weights(const std::vector<E>& w, bool inverse) {
        size_t n = w.size();
        std::vector<F> c0(n), c1(n);
        F b[2];
        for (size_t i = 0; i < n; i++) { w[i].as_bases(b); c0[i] = b[0]; c1[i] = E::DEGREE > 1 ? b[1] : F::zero(); }
        ntt_naive_order(c0, inverse);
        if (E::DEGREE > 1) ntt_naive_order(c1, inverse);
        std::vector<E> A(n);
        for (size_t i = 0; i < n; i++) { b[0] = c0[i]; b[1] = c1[i]; A[i] = E::from_bases(b); }
        return A;
    }

    // sumcheck of sum_x t0[x] * prod_k tabs[k][x] (degree 1 + #tabs), all tables over E; returns point, final evals
    static void product_sumcheck(std::vector<std::vector<E>> tabs, E claim, Transcript<F>& tr, std::vector<E>* point, std::vector<E>* finals,
                                 size_t capture_len = 0, std::vector<E>* captured = nullptr, size_t capture_tab = 1) {
        const int d = (int)tabs.size();
        size_t n = tabs[0].size();
        point->clear();
        while (n > 1) {
            if (captured && n == capture_len) *captured = tabs[capture_tab];
            const size_t h = n / 2;
            std::vector<E> ev(d + 1, E::zero());
#pragma omp parallel if (h >= 2048)
            {
                E loc[5] = {E::zero(), E::zero(), E::zero(), E::zero(), E::zero()};
#pragma omp for schedule(static) nowait
                for (size_t b = 0; b < h; b++) {
                    E lo[4], df[4];
                    for (int k = 0; k < d; k++) { lo[k] = tabs[k][2 * b]; df[k] = tabs[k][2 * b + 1] - lo[k]; }
                    for (int x = 0; x <= d; x++) {
                        E p = lo[0];
                        for (int k = 1; k < d; k++) p *= lo[k];
                        for (int k = 0; k < d; k++) lo[k] += df[k];
                        loc[x] += p;
                    }
                }
#pragma omp critical
                for (int x = 0; x <= d; x++) ev[x] += loc[x];
            }
            if (assumptions().a3_h1 == 0) ev[1] = claim - ev[0];
            std::vector<E> co = interpolate_coeffs<E, F>(ev);
            if (assumptions().a3_wire == 0) { tr.write(co[0]); for (int i = 2; i <= d; i++) tr.write(co[i]); }
            else { tr.write(ev[0]); for (int i = 2; i <= d; i++) tr.write(ev[i]); }
            E r = tr.squeeze();
            claim = horner(co, r);
            for (auto& t : tabs) {
                std::vector<E> nx(h);
#pragma omp parallel for schedule(static) if (h >= 4096)
                for (size_t b = 0; b < h; b++) nx[b] = t[2 * b] + r * (t[2 * b + 1] - t[2 * b]);
                t.swap(nx);
            }
            point->push_back(r);
            n = h;
        }
        if (captured && capture_len == 1) *captured = tabs[capture_tab];
        finals->resize(d);
        for (int k = 0; k < d; k++) (*finals)[k] = tabs[k][0];
    }
    static void product_sumcheck_verify(int d, int num_vars, E claim, Transcript<F>& tr, std::vector<E>* point, E* final_claim) {
        point->clear();
        for (int round = 0; round < num_vars; round++) {
            std::vector<E> m(d + 1);
            m[0] = tr.read(); for (int i = 2; i <= d; i++) m[i] = tr.read();
            E r = tr.squeeze();
            if (assumptions().a3_wire == 0) { E s = m[0].dbl(); for (int i = 2; i <= d; i++) s += m[i]; m[1] = claim - s; claim = horner(m, r); }
            else { m[1] = claim - m[0]; claim = lagrange_eval<E, F>(m, r); }
            point->push_back(r);
        }
        *final_claim = claim;
    }
    static std::vector<E> lift_vec(const std::vector<F>& v) { std::vector<E> r(v.size()); for (size_t i = 0; i < v.size(); i++) r[i] = E::from_base(v[i]); return r; }
    static int log2sz(size_t n) { int l = 0; while (((size_t)1 << l) < n) l++; return l; }

    // ---- one node's claim reduction (prover). Returns the claims pushed to each predecessor.
    std::vector<std::vector<EvalClaim<F>>> prove_node(int id, const std::vector<EvalClaim<F>>& claims, const std::vector<std::vector<F>>& val,
                                                      Transcript<F>& tr) const {
        const auto& nd = nodes[id];
        std::vector<std::vector<EvalClaim<F>>> out(nd.preds.size());
        if (nd.kind == NODE_LASSO) {
            std::vector<E> r; E s;
            nd.lasso->prove_claim_reduction(val[nd.preds.at(0)], tr, &r, &s);
            out[0].push_back({r, s});
            return out;
        }
        E alpha = E::one();
        if (claims.size() > 1) alpha = tr.squeeze();
        E combined = E::zero();
        { E p = E::one(); for (auto& c : claims) { combined += p * c.value; p *= alpha; } }
        std::vector<E> w = combined_eq(claims, alpha, nd.out_len());
        std::vector<E> pt, fin;
        if (nd.kind == NODE_FFT) {
            std::vector<E> A = fft_weights(w, nd.fft_inverse);
            product_sumcheck({A, lift_vec(val[nd.preds.at(0)])}, combined, tr, &pt, &fin);
            tr.write(fin[1]);
            out[0].push_back({pt, fin[1]});
        } else if (nd.elementwise_mul()) {
            product_sumcheck({w, lift_vec(val[nd.preds[0]]), lift_vec(val[nd.preds[1]])}, combined, tr, &pt, &fin);
            tr.write(fin[1]); tr.write(fin[2]);
            out[0].push_back({pt, fin[1]});
            out[1].push_back({pt, fin[2]});
        } else if (nd.linear()) {
            Reduction R = linear_reduction(nd, w, &val);
            std::vector<E> cap;
            product_sumcheck({R.A, lift_vec(R.X)}, combined - R.constant, tr, &pt, &fin, R.a_pad, &cap, 1);
            std::vector<E> lo(pt.begin(), pt.begin() + log2sz(R.n_in));
            for (int k = 0; k < nd.arity; k++) { tr.write(cap[k]); out[k].push_back({lo, cap[k]}); }
        } else {
            throw OracleError("prove_node: gate shape outside the restated engine (only linear layers and the element-wise product)");
        }
        return out;
    }
    std::vector<std::vector<EvalClaim<F>>> verify_node(int id, const std::vector<EvalClaim<F>>& claims, Transcript<F>& tr) const {
        const auto& nd = nodes[id];
        std::vector<std::vector<EvalClaim<F>>> out(nd.preds.size());
        if (nd.kind == NODE_LASSO) {
            std::vector<E> r; E s;
            nd.lasso->verify_claim_reduction(tr, &r, &s);
            out[0].push_back({r, s});
            return out;
        }
        E alpha = E::one();
        if (claims.size() > 1) alpha = tr.squeeze();
        E combined = E::zero();
        { E p = E::one(); for (auto& c : claims) { combined += p * c.value; p *= alpha; } }
        std::vector<E> w = combined_eq(claims, alpha, nd.out_len());
        std::vector<E> pt; E fc;
        if (nd.kind == NODE_FFT) {
            product_sumcheck_verify(2, nd.log2_size, combined, tr, &pt, &fc);
            E in_eval = tr.read();
            E a = mle_evaluate_ext(fft_weights(w, nd.fft_inverse), pt);
            if (a * in_eval != fc) throw OracleError("InvalidSumCheck: FFT layer final evaluation mismatch");
            out[0].push_back({pt, in_eval});
        } else if (nd.elementwise_mul()) {
            product_sumcheck_verify(3, log2sz(nd.out_len()), combined, tr, &pt, &fc);
            E a = tr.read(), b = tr.read();
            if (mle_evaluate_ext(w, pt) * a * b != fc) throw OracleError("InvalidSumCheck: product layer final evaluation mismatch");
            out[0].push_back({pt, a});
            out[1].push_back({pt, b});
        } else if (nd.linear()) {
            Reduction R = linear_reduction(nd, w, nullptr);
            product_sumcheck_verify(2, log2sz(R.a_pad * R.n_in), combined - R.constant, tr, &pt, &fc);
            std::vector<E> lo(pt.begin(), pt.begin() + log2sz(R.n_in)), hi(pt.begin() + log2sz(R.n_in), pt.end());
            std::vector<E> eqhi = eq_xy(hi);
            E x = E::zero();
            for (int k = 0; k < nd.arity; k++) { E e = tr.read(); x += eqhi[k] * e; out[k].push_back({lo, e}); }
            if (mle_evaluate_ext(R.A, pt) * x != fc) throw OracleError("InvalidSumCheck: linear layer final evaluation mismatch");
        } else {
            throw OracleError("verify_node: unsupported gate shape");
        }
        return out;
    }

    std::vector<int> output_nodes() const { std::vector<int> o; for (size_t i = 0; i < nodes.size(); i++) if (nodes[i].succs.empty() && nodes[i].kind != NODE_INPUT) o.push_back((int)i); return o; }

    // ---- prove_gkr / verify_gkr (call sites sk_encryption_circuit.rs:455-457, :509-510): reverse topological order;
    // returns the claims that reached the input nodes, in insertion order
    std::vector<std::vector<EvalClaim<F>>> prove_gkr(const std::vector<std::vector<F>>& val, const std::vector<EvalClaim<F>>& output_claims, Transcript<F>& tr) const {
        std::vector<std::vector<EvalClaim<F>>> claims(nodes.size());
        auto outs = output_nodes();
        if (outs.size() != output_claims.size()) throw OracleError("prove_gkr: output claim count mismatch");
        for (size_t i = 0; i < outs.size(); i++) claims[outs[i]].push_back(output_claims[i]);
        auto order = topo_order();
        for (size_t oi = order.size(); oi-- > 0;) {
            const int id = order[oi];
            if (nodes[id].kind == NODE_INPUT) continue;
            auto sub = prove_node(id, claims[id], val, tr);
            for (size_t k = 0; k < sub.size(); k++) for (auto& c : sub[k]) claims[nodes[id].preds[k]].push_back(c);
        }
        std::vector<std::vector<EvalClaim<F>>> r;
        for (size_t id = 0; id < nodes.size(); id++) if (nodes[id].kind == NODE_INPUT) r.push_back(claims[id]);
        return r;
    }
    std::vector<std::vector<EvalClaim<F>>> verify_gkr(const std::vector<EvalClaim<F>>& output_claims, Transcript<F>& tr) const {
        std::vector<std::vector<EvalClaim<F>>> claims(nodes.size());
        auto outs = output_nodes();
        for (size_t i = 0; i < outs.size(); i++) claims[outs[i]].push_back(output_claims[i]);
        auto order = topo_order();
        for (size_t oi = order.size(); oi-- > 0;) {
            const int id = order[oi];
            if (nodes[id].kind == NODE_INPUT) continue;
            auto sub = verify_node(id, claims[id], tr);
            for (size_t k = 0; k < sub.size(); k++) for (auto& c : sub[k]) claims[nodes[id].preds[k]].push_back(c);
        }
        std::vector<std::vector<EvalClaim<F>>> r;
        for (size_t id = 0; id < nodes.size(); id++) if (nodes[id].kind == NODE_INPUT) r.push_back(claims[id]);
        return r;
    }
};

// ---------------------------------------------------------------- BfvEncrypt (bfv-gkr/src/sk_encryption_circuit.rs)
template <class F> struct BfvEncrypt {
    typedef typename ExtOf<F>::type E;
    BfvParams<F> P;
    int n_log2;
    Circuit<F> circuit;
    Preprocessing pp;
    int lasso_num_vars = 0;

    static GkrNode<F> input(int log2_size, int reps) { GkrNode<F> n; n.kind = NODE_INPUT; n.log2_size = log2_size; n.num_reps = reps; return n; }
    static GkrNode<F> vanilla(int arity, int log2_sub, std::vector<VanillaGate<F>> gates, int reps) {
        GkrNode<F> n; n.kind = NODE_VANILLA; n.arity = arity; n.log2_sub_input = log2_sub; n.gates = std::move(gates); n.num_reps = reps; return n;
    }
    static GkrNode<F> fft(int log2_size, bool inverse) { GkrNode<F> n; n.kind = NODE_FFT; n.log2_size = log2_size; n.fft_inverse = inverse; return n; }
    static VanillaGate<F> relay_mul_const(int in, size_t w, F c) { VanillaGate<F> g; g.adds.push_back({c, in, w}); return g; }      // :525-527
    static VanillaGate<F> relay_add_const(int in, size_t w, F c) { VanillaGate<F> g; g.has_const = true; g.c = c; g.adds.push_back({F::one(), in, w}); return g; }  // :529-531

    // setup (:319-349) + configure (:351-363, :86-293)
    explicit BfvEncrypt(const BfvParams<F>& params) : P(params) {
        const int L = P.log2_size, K = P.K;
        n_log2 = L - 1;
        const size_t N2 = (size_t)1 << L;
        std::vector<uint64_t> bounds = {P.s_bound * 2 + 1, P.e_bound * 2 + 1, P.k1_bound * 2 + 1};
        for (int i = 0; i < K; i++) bounds.push_back(P.r1_bounds[i] * 2 + 1);
        for (int i = 0; i < K; i++) bounds.push_back(P.r2_bounds[i] * 2 + 1);
        pp = Preprocessing::preprocess(bounds, 4, 16);
        auto& c = circuit;
        int s = c.insert(input(L, 1)), e = c.insert(input(L, 1)), k1 = c.insert(input(L, 1));
        std::vector<VanillaGate<F>> g;
        for (int i = 0; i < K; i++) for (size_t j = 0; j < N2; j++) g.push_back(VanillaGate<F>::relay(0, j));
        int es = c.insert(vanilla(1, L, g, 1));
        g.clear();
        for (int i = 0; i < K; i++) for (size_t j = 0; j < N2; j++) g.push_back(relay_mul_const(0, j, P.k0is[i]));
        int k1kis = c.insert(vanilla(1, L, g, 1));
        c.connect(e, es); c.connect(k1, k1kis);
        std::vector<int> ais, r1is;
        for (int i = 0; i < K; i++) ais.push_back(c.insert(input(L, 1)));
        for (int i = 0; i < K; i++) r1is.push_back(c.insert(input(L, 1)));
        g.clear();
        for (int i = 0; i < K; i++) for (size_t j = 0; j < N2; j++) g.push_back(relay_mul_const(i, j, P.qis[i]));
        int r1iqis = c.insert(vanilla(K, L, g, 1));
        for (int i = 0; i < K; i++) c.connect(r1is[i], r1iqis);
        int r2is = c.insert(input(n_log2, K));
        int r2_log2 = n_log2 + ilog2_u64(K);
        std::vector<int> chunks;
        for (size_t start = 0; start < ((size_t)1 << r2_log2); start += N2) {
            g.clear();
            for (size_t j = start; j < std::min(start + N2, (size_t)1 << r2_log2); j++) g.push_back(VanillaGate<F>::relay(0, j));
            g.resize(N2, VanillaGate<F>::constant(F::zero()));
            int nd = c.insert(vanilla(1, r2_log2, g, 1));
            c.connect(r2is, nd);
            chunks.push_back(nd);
        }
        g.clear();
        {
            std::vector<uint64_t> shift;
            for (int i = 0; i < K; i++) shift.push_back(P.r1_bounds[i]);
            for (size_t i = 0; i < chunks.size(); i++) shift.push_back(P.r2_bounds[0]);
            shift.push_back(P.s_bound); shift.push_back(P.e_bound); shift.push_back(P.k1_bound);
            for (size_t i = 0; i < shift.size(); i++) for (size_t j = 0; j < N2; j++) g.push_back(relay_add_const((int)i, j, F::from_u64(shift[i])));
        }
        int lasso_in = c.insert(vanilla((int)chunks.size() + K + 3, L, g, 1));
        // lookups (:182-210)
        std::vector<int> rows;
        auto push = [&](uint64_t bound, size_t cnt) { int li = pp.lookup_id_to_index.at(RangeLookup{bound}.id()); rows.insert(rows.end(), cnt, li); };
        const size_t r2i_len = K == 1 ? N2 : N2 / 2;
        for (int i = 0; i < K; i++) push(P.r1_bounds[i] * 2 + 1, N2);
        for (int i = 0; i < K; i++) push(P.r2_bounds[i] * 2 + 1, r2i_len);
        push(P.s_bound * 2 + 1, N2); push(P.e_bound * 2 + 1, N2); push(P.k1_bound * 2 + 1, N2);
        lasso_num_vars = 0; while (((size_t)1 << lasso_num_vars) < rows.size()) lasso_num_vars++;
        GkrNode<F> ln; ln.kind = NODE_LASSO; ln.lasso = std::make_shared<LassoNode<F>>(pp, lasso_num_vars, rows);
        int lasso = c.insert(ln);
        for (int i = 0; i < K; i++) c.connect(r1is[i], lasso_in);
        for (int ch : chunks) c.connect(ch, lasso_in);
        c.connect(s, lasso_in); c.connect(e, lasso_in); c.connect(k1, lasso_in);
        c.connect(lasso_in, lasso);
        int s_eval = c.insert(fft(L, false));
        c.connect(s, s_eval);
        g.clear();
        for (size_t j = 0; j < N2; j++) g.push_back(VanillaGate<F>::relay(0, j));
        int s_copy = c.insert(vanilla(1, L, g, 1));
        c.connect(s_eval, s_copy);
        g.clear();
        for (int i = 0; i < K; i++) for (size_t j = 0; j < N2; j++) g.push_back(VanillaGate<F>::relay(i, j));
        int sai_par = c.insert(vanilla(K, L, g, 1));
        for (int i = 0; i < K; i++) {
            g.clear();
            for (size_t j = 0; j < N2; j++) g.push_back(VanillaGate<F>::mul(0, j, 1, j));
            int ai_eval = c.insert(fft(L, false));
            int sai_eval = c.insert(vanilla(2, L, g, 1));
            int sai = c.insert(fft(L, true));
            c.connect(ais[i], ai_eval);
            c.connect(s_copy, sai_eval); c.connect(ai_eval, sai_eval);
            c.connect(sai_eval, sai);
            c.connect(sai, sai_par);
        }
        g.clear();
        {
            const size_t r2i_size = ((size_t)1 << n_log2) - 1;
            for (size_t i = 0; i < r2i_size; i++) g.push_back(VanillaGate<F>::relay(0, i));
            g.push_back(VanillaGate<F>::constant(F::zero()));
            for (size_t i = 0; i < r2i_size; i++) g.push_back(VanillaGate<F>::relay(0, i));
            g.push_back(VanillaGate<F>::constant(F::zero()));
        }
        int cyclo = c.insert(vanilla(1, n_log2, g, K));
        g.clear();
        for (size_t j = 0; j < N2; j++) g.push_back(VanillaGate<F>::sum({{0, j}, {1, j}, {2, j}, {3, j}, {4, j}}));
        int sum = c.insert(vanilla(5, L, g, K));
        c.connect(r2is, cyclo);
        c.connect(sai_par, sum); c.connect(es, sum); c.connect(k1kis, sum); c.connect(r1iqis, sum); c.connect(cyclo, sum);
    }
    int ct0is_log2_size() const { return P.log2_size + ilog2_u64(P.K); }  // :519-522

    // inputs in the order get_inputs returns them (:408): s, e, k1, ais.., r1is.., r2is — which is also insertion order
    // of the input nodes except that r2is is inserted after the r1is (same order) -> identical.
    std::vector<uint8_t> prove(const std::vector<std::vector<F>>& inputs, const std::vector<F>& ct0is,
                               std::vector<std::vector<EvalClaim<F>>>* input_claims = nullptr) const {
        Transcript<F> tr;
        auto val = circuit.evaluate(inputs);                                   // :442
        std::vector<E> point = tr.squeeze_n(ct0is_log2_size());                // :445
        E value = mle_evaluate<E, F>(ct0is, point);                            // :446
        std::vector<EvalClaim<F>> oc = {{{}, E::zero()}, {point, value}};      // :450
        auto ic = circuit.prove_gkr(val, oc, tr);                              // :455-457
        if (input_claims) *input_claims = ic;
        return tr.stream;
    }
    // verify (:462-517): recompute the output claim, verify_gkr, check every input claim against the inputs
    void verify(const std::vector<std::vector<F>>& inputs, const std::vector<F>& ct0is, const uint8_t* proof, size_t len) const {
        Transcript<F> tr(proof, len);
        std::vector<E> point = tr.squeeze_n(ct0is_log2_size());
        E value = mle_evaluate<E, F>(ct0is, point);
        std::vector<EvalClaim<F>> oc = {{{}, E::zero()}, {point, value}};
        auto ic = circuit.verify_gkr(oc, tr);
        if (tr.rd_pos != len) throw OracleError("verify: trailing bytes in proof");
        if (ic.size() != inputs.size()) throw OracleError("verify: input count mismatch");
        for (size_t i = 0; i < inputs.size(); i++)
            for (auto& c : ic[i])
                if (mle_evaluate<E, F>(inputs[i], c.point) != c.value) throw OracleError("verify: input claim does not match the input (sk_encryption_circuit.rs:515)");
    }
};

}  // namespace hgo
