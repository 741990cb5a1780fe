// extern "C" boundary (include/hg_b200.h). Translates handles + limb arrays to the templated C++/CUDA implementation
// and turns every exception into an error code + message.
#include "../../include/hg_b200.h"

#include <cstring>
#include <memory>
#include <string>
#include <type_traits>
#include <variant>
#include <vector>

#include <map>

#include "bfv_circuit.hpp"
#include "gkr_dev.cuh"
#include "prover.cuh"
#include "lasso_verify.hpp"
#include "gkr_verify.hpp"
#include "witness_gen.cuh"

using namespace hg;

namespace {
thread_local std::string g_err;
int fail(const std::string& m) { g_err = m; return 1; }
#define HG_TRY(...)                                                             \
    try { __VA_ARGS__; return 0; }                                              \
    catch (const std::exception& e) { cudaGetLastError(); return fail(e.what()); } \
    catch (...) { cudaGetLastError(); return fail("unknown error"); }

template <class FP> __global__ void k_selftest(int op, const typename FP::X* a, const typename FP::X* b, size_t n, typename FP::X* out) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    typename FP::X x = a[i], y = b[i], z;
    if (op == 0) z = FP::x_add(x, y);
    else if (op == 1) z = FP::x_sub(x, y);
    else z = FP::x_mul(x, y);
    out[i] = z;
}
}  // namespace

template <class FP> __global__ void k_field_encode(typename FP::B* p, size_t n, int decode) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if constexpr (FP::FIELD_ID == 1) {
        fr v = p[i];
        if (decode) { u64 t[4]; fr_to_canonical(v, t); p[i] = fr_make(t[0], t[1], t[2], t[3]); }
        else p[i] = fr_from_canonical(v.l);
    }
}

// acc[i] = sum over parts of parts[r][i] in the extension field (the message buffers of the devices of one sharded proof)
template <class FP> __global__ void k_shard_merge(const typename FP::X* __restrict__ parts, int world, size_t n, typename FP::X* __restrict__ acc) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    typename FP::X s = parts[i];
    for (int r = 1; r < world; r++) s = FP::x_add(s, parts[(size_t)r * n + i]);
    acc[i] = s;
}

// ---- fields. Every handle holds its object typed by its field; the templates behind them are instantiated for GlField
// (Goldilocks / GoldilocksExt2) and FrField (BN254 Fr, E = F). with_field is the one place a field id becomes a type.
template <class F> decltype(auto) with_field(int field_id, F&& f) {
    if (field_id == HG_FIELD_GOLDILOCKS) return f(GlField{});
    if (field_id == HG_FIELD_BN254) return f(FrField{});
    throw std::runtime_error("unknown field id");
}
// the field of a handle's object (Keccak256Transcript<FP>, LassoNodeDev<FP>, GkrCircuitDev<FP>, GkrVerifierHost<FP>)
template <class T> struct field_of;
template <template <class> class H, class FP> struct field_of<H<FP>> { typedef FP type; };
template <class T> using field_t = typename field_of<std::remove_cv_t<std::remove_reference_t<T>>>::type;
// messages of a sharded proof cross the boundary in the device representation, as 64-bit words
template <class FP> constexpr size_t XW = sizeof(typename FP::X) / sizeof(uint64_t);

// per-field work state of a context
template <class FP> struct FieldState {
    typedef typename FP::X X;
    std::unique_ptr<NttEngine<FP>> engine;  // created on first use
    NttEngine<FP>* eng(DeviceCtx* ctx) { if (!engine) engine.reset(new NttEngine<FP>(ctx)); return engine.get(); }
    // hg_bfv_witness_generate
    DevBuf<signed char> wg_s, wg_e;
    DevBuf<int> wg_k1;
    DevBuf<long long> wg_a;
    DevBuf<i128> wg_hat;
    DevBuf<WitGenStatus> wg_st;
    // hg_mle_eval_batch
    DevBuf<X> mle_pt, mle_eq, mle_partials, mle_out;
    DevBuf<unsigned> mle_counters;
    PinnedBuf<X> mle_hpt;
};

struct hg_ctx {
    DeviceCtx dev;
    int field_id;
    WireOptions wire;
    std::variant<std::monostate, FieldState<GlField>, FieldState<FrField>> state;  // monostate once hg_ctx_destroy released it
};
struct InputClaimErased { std::vector<uint64_t> point; std::vector<uint64_t> value; size_t nvars; };
struct hg_circuit {
    template <class C, class... A> hg_circuit(hg_ctx* x, int field, std::in_place_type_t<C> kind, A&&... a) : ctx(x), field_id(field), c(kind, std::forward<A>(a)...) {}
    hg_ctx* ctx;  // nullptr: a host-only circuit description (hg_circuit_new_host), usable for hg_gkr_verify only
    int field_id;
    std::variant<GkrCircuitDev<GlField>, GkrCircuitDev<FrField>, GkrVerifierHost<GlField>, GkrVerifierHost<FrField>> c;
    std::vector<std::vector<InputClaimErased>> input_claims;  // per input node, from the last prove / verify
    DevBuf<unsigned char> host_arena;  // hg_circuit_evaluate_host: the circuit's own copy of the inputs
};
static void circuit_use_device(hg_circuit* c) {
    if (!c->ctx) throw std::runtime_error("this circuit is a host-only description (hg_circuit_new_host): it has no device, only hg_gkr_verify runs on it");
    HG_CUDA(cudaSetDevice(c->ctx->dev.device));
}
struct hg_buf {
    void* p = nullptr;
    size_t bytes = 0;
    int device = 0;
};
struct hg_transcript {
    std::variant<Keccak256Transcript<GlField>, Keccak256Transcript<FrField>> t;
};
struct hg_lasso_pp {
    LassoPreprocessing pp;
    std::vector<uint64_t> lookup_bounds;  // in preprocessing order
};
struct hg_lasso_node {
    template <class FP> hg_lasso_node(hg_ctx* c, FP, const LassoPreprocessing& pp, size_t num_vars, const std::vector<uint8_t>& rows)
        : ctx(c), node(std::in_place_type<LassoNodeDev<FP>>, &c->dev, pp, (int)num_vars, rows), log2_input_size(std::max<size_t>(num_vars, ilog2u(pp.M))) {}  // lasso.rs:45-47
    hg_ctx* ctx;
    std::variant<LassoNodeDev<GlField>, LassoNodeDev<FrField>> node;
    DevBuf<unsigned char> staging;  // host inputs on their way to the device
    size_t log2_input_size;
};

// ---- the typed object of a handle, for a field the caller already knows (from another handle): a handle of another field is an error
template <class T, class V> T& typed_as(V& v, const char* what) {
    if (T* p = std::get_if<T>(&v)) return *p;
    throw std::runtime_error(std::string(what) + " belongs to another field");
}
template <class FP> Keccak256Transcript<FP>& typed(hg_transcript* t) { return typed_as<Keccak256Transcript<FP>>(t->t, "transcript"); }
template <class FP> LassoNodeDev<FP>& typed(hg_lasso_node* n) { return typed_as<LassoNodeDev<FP>>(n->node, "lasso node"); }
template <class FP> FieldState<FP>& typed(hg_ctx* c) { return typed_as<FieldState<FP>>(c->state, "context"); }
// f(the circuit as K<FP>): K = GkrCircuitDev for a device circuit, GkrVerifierHost for a host-only description. The caller
// has checked which of the two the circuit is.
template <template <class> class K, class H, class F> decltype(auto) with_kind(H* c, F&& f) {
    return with_field(c->field_id, [&](auto fp) -> decltype(auto) { return f(std::get<K<decltype(fp)>>(c->c)); });
}

// ---- limbs across the boundary
static WireOptions wire_options(const int* options3) {  // NULL: the defaults
    WireOptions wo;
    if (options3) { wo.a3_wire = options3[0]; wo.a3_h1 = options3[1]; wo.a5_ascending = options3[2]; }
    return wo;
}
// an extension-field point and value to limbs; a NULL output is skipped
template <class FP> void claim_to_limbs(const std::vector<typename FP::X>& pt, const typename FP::X& val, uint64_t* out_point, uint64_t* out_value) {
    if (out_point) for (size_t i = 0; i < pt.size(); i++) FP::x_to_limbs(pt[i], out_point + FP::X_LIMBS * i);
    if (out_value) FP::x_to_limbs(val, out_value);
}
// output claims from limbs: claim i has lens[i] coordinates (the points back to back in pts) and one value in vals
template <class FP, class Claim> std::vector<Claim> claims_from_limbs(size_t n_claims, const size_t* lens, const uint64_t* pts, const uint64_t* vals) {
    std::vector<Claim> oc(n_claims);
    size_t off = 0;
    for (size_t i = 0; i < n_claims; i++) {
        for (size_t k = 0; k < lens[i]; k++) oc[i].point.push_back(FP::x_from_limbs(pts + FP::X_LIMBS * (off + k)));
        off += lens[i];
        oc[i].value = FP::x_from_limbs(vals + FP::X_LIMBS * i);
    }
    return oc;
}
// the input claims a prove / verify returned, as limbs (hg_gkr_input_claim reads them without knowing the field)
template <class FP, class Claim> void set_input_claims(hg_circuit* c, const std::vector<std::vector<Claim>>& res) {
    c->input_claims.clear();
    for (auto& v : res) {
        std::vector<InputClaimErased> e;
        for (auto& ic : v) {
            InputClaimErased x;
            x.nvars = ic.point.size();
            x.point.resize(ic.point.size() * FP::X_LIMBS);
            x.value.resize(FP::X_LIMBS);
            claim_to_limbs<FP>(ic.point, ic.value, x.point.data(), x.value.data());
            e.push_back(x);
        }
        c->input_claims.push_back(e);
    }
}
// a Lasso node's inputs on the device: host inputs are uploaded to the node's staging buffer and, for BN254, brought to the
// device representation, asynchronously on the context's stream
template <class FP> const typename FP::B* stage(hg_lasso_node* node, const void* inputs, size_t n_inputs, bool on_device) {
    typedef typename FP::B B;
    if (on_device) return (const B*)inputs;
    DeviceCtx* dev = &node->ctx->dev;
    if (node->staging.n < n_inputs * sizeof(B)) node->staging.alloc(n_inputs * sizeof(B));
    B* p = (B*)node->staging.p;
    HG_CUDA(cudaMemcpyAsync(p, inputs, n_inputs * sizeof(B), cudaMemcpyHostToDevice, dev->stream));
    if (FP::FIELD_ID == 1) { k_field_encode<FP><<<(unsigned)((n_inputs + 255) / 256), 256, 0, dev->stream>>>(p, n_inputs, 0); HG_LAUNCH_CHECK(); }
    return p;
}
template <class... A> hg_transcript* new_transcript(int field_id, const A&... a) {  // a: Keccak256Transcript's constructor arguments
    return with_field(field_id, [&](auto fp) { return new hg_transcript{Keccak256Transcript<decltype(fp)>(a...)}; });
}
static const std::vector<uint8_t>& proof_bytes(const hg_transcript* t) {
    return std::visit([](auto& tr) -> const std::vector<uint8_t>& { return tr.proof(); }, t->t);
}
static hg_lasso_node* new_lasso_node(hg_ctx* ctx, const hg_lasso_pp* pp, size_t num_vars, const std::vector<uint8_t>& rows) {
    return with_field(ctx->field_id, [&](auto fp) { return new hg_lasso_node(ctx, fp, pp->pp, num_vars, rows); });
}

// ---- entry-point bodies generic over the field (the extern "C" functions below dispatch to them)

// hg_circuit_evaluate_host. The circuit's own copy of the inputs (allocated once): host vectors are uploaded and, for BN254,
// brought to the device representation, all asynchronously on the context's stream; evaluate follows in stream order
template <class FP> void evaluate_host(hg_circuit* hc, GkrCircuitDev<FP>& c, const void* const* in, const size_t* n_elems, size_t n) {
    typedef typename FP::B B;
    DeviceCtx* dev = &hc->ctx->dev;
    const std::vector<size_t> lens = c.input_lens();
    if (n != lens.size()) throw std::runtime_error("evaluate: wrong number of inputs");
    size_t total = 0;
    for (size_t i = 0; i < n; i++) {
        if (n_elems[i] != lens[i]) throw std::runtime_error("evaluate: input length does not match the input node");
        total += lens[i];
    }
    if (hc->host_arena.n != total * sizeof(B)) hc->host_arena.alloc(total * sizeof(B));
    B* arena = (B*)hc->host_arena.p;  // all inputs back to back, in input-node order
    std::vector<const B*> v;
    // host vectors that are adjacent in memory (one pinned block, as a caller that wants speed lays them out) go in one copy.
    // Adjacent addresses can also belong to two separate page-locked allocations, for which one copy is invalid: then the
    // run is copied vector by vector.
    size_t off = 0;
    std::vector<size_t> offs(n);
    for (size_t i = 0; i < n; i++) { offs[i] = off; v.push_back(arena + off); off += lens[i]; }
    for (size_t i = 0; i < n;) {
        size_t k = i + 1, run_len = lens[i];
        while (k < n && (const char*)in[k] == (const char*)in[i] + run_len * sizeof(B)) { run_len += lens[k]; k++; }
        cudaError_t e = cudaMemcpyAsync(arena + offs[i], in[i], run_len * sizeof(B), cudaMemcpyHostToDevice, dev->stream);
        if (e != cudaSuccess && k > i + 1) {
            cudaGetLastError();
            for (size_t q = i; q < k; q++) HG_CUDA(cudaMemcpyAsync(arena + offs[q], in[q], lens[q] * sizeof(B), cudaMemcpyHostToDevice, dev->stream));
        } else if (e != cudaSuccess) {
            HG_CUDA(e);
        }
        i = k;
    }
    if (FP::FIELD_ID == 1) { k_field_encode<FP><<<(unsigned)((total + 255) / 256), 256, 0, dev->stream>>>(arena, total, 0); HG_LAUNCH_CHECK(); }
    c.evaluate(v);
}

// hg_sumcheck_prove
template <class FP> void sumcheck_prove(hg_ctx* ctx, int arity, size_t n_terms, size_t num_vars, const uint64_t* coeffs_ext, const void* d_tables,
                                        const uint64_t* claim_ext, hg_transcript* t, int mode, uint64_t* out_point, uint64_t* out_evals) {
    typedef typename FP::B B;
    typedef typename FP::X X;
    DeviceCtx* dev = &ctx->dev;
    const WireOptions& wo = ctx->wire;
    if (arity != 1 && arity != 2) throw std::runtime_error("arity must be 1 or 2");
    if (num_vars < 1 || num_vars > 30) throw std::runtime_error("num_vars out of range");
    Keccak256Transcript<FP>& tr = typed<FP>(t);
    const size_t n = (size_t)1 << num_vars, ntab = n_terms * arity;
    DevBuf<X> coeffs, bufA, bufB, partials;
    DevBuf<unsigned> counters;
    coeffs.alloc(n_terms);
    std::vector<X> hc(n_terms);
    for (size_t i = 0; i < n_terms; i++) hc[i] = FP::x_from_limbs(coeffs_ext + FP::X_LIMBS * i);
    HG_CUDA(cudaMemcpyAsync(coeffs.p, hc.data(), n_terms * sizeof(X), cudaMemcpyHostToDevice, dev->stream));
    HG_CUDA(cudaStreamSynchronize(dev->stream));  // hc is a stack temporary
    bufA.alloc(std::max<size_t>(ntab * (n / 2), ntab));
    bufB.alloc(std::max<size_t>(ntab * (n / 4), ntab));
    ScScratch sc;
    sc.max_blocks = dev->sm_count * 8;
    partials.alloc((size_t)sc.max_blocks * 4);
    counters.alloc(4);
    HG_CUDA(cudaMemset(counters.p, 0, counters.bytes()));
    sc.partials = partials.p; sc.counters = counters.p;
    Channel<FP> ch(dev, num_vars + 1, 4 * num_vars + ntab + 4);
    Keccak256Transcript<FP>* trp = &tr;
    ch.begin(trp, (mode == HG_MODE_INTERACTIVE || !trp->prefetch_legal()) ? kModeInteractive : kModePrefetch, num_vars);
    auto st = std::make_shared<ScHostState<FP>>();
    st->claim = FP::x_from_limbs(claim_ext);
    size_t first = 0, eo = 0;
    if (arity == 1) sumcheck_dev<FP, 1>(dev, KC_SC_COLL, ch, wo, (const B*)d_tables, n, (int)n_terms, coeffs.p, bufA.p, bufB.p, sc, st, &first, &eo);
    else sumcheck_dev<FP, 2>(dev, KC_SC_GP, ch, wo, (const B*)d_tables, n, (int)n_terms, coeffs.p, bufA.p, bufB.p, sc, st, &first, &eo);
    ch.flush();
    if (out_point) for (size_t i = 0; i < num_vars; i++) FP::x_to_limbs(ch.chal(first + i), out_point + FP::X_LIMBS * i);
    if (out_evals) for (size_t i = 0; i < ntab; i++) FP::x_to_limbs(ch.msg(eo + i), out_evals + FP::X_LIMBS * i);
}

// hg_mle_eval_batch
template <class FP> void mle_eval_batch(hg_ctx* ctx, const void* d_tables, size_t n_tables, size_t stride, size_t num_vars, const uint64_t* point_ext, uint64_t* out_ext) {
    typedef typename FP::B B;
    typedef typename FP::X X;
    DeviceCtx* dev = &ctx->dev;
    FieldState<FP>& fs = typed<FP>(ctx);
    const size_t n = (size_t)1 << num_vars;
    // k_dot_eq reads a table four entries at a time with 16-byte vector loads from its first entry on (num_vars >= 2)
    if (num_vars >= 2 && (((uintptr_t)d_tables | (stride * sizeof(B))) & 15) != 0)
        throw std::runtime_error("hg_mle_eval_batch: every table must start 16-byte aligned (d_tables and stride * element size)");
    cudaStream_t s = dev->stream;
    // work buffers persist across calls (a cudaMalloc / cudaFree pair per buffer costs more than the evaluation)
    DevBuf<X>&pt = fs.mle_pt, &eq = fs.mle_eq, &partials = fs.mle_partials, &out = fs.mle_out;
    DevBuf<unsigned>& counters = fs.mle_counters;
    PinnedBuf<X>& hpt = fs.mle_hpt;
    auto grow = [&](auto& buf, size_t need) { if (buf.n < need) { HG_CUDA(cudaStreamSynchronize(s)); buf.alloc(need + need / 2); } };
    const size_t np = std::max<size_t>(num_vars, 1);
    grow(pt, np);
    if (hpt.n < np + n_tables) hpt.alloc(2 * (np + n_tables));
    for (size_t i = 0; i < num_vars; i++) hpt.p[i] = FP::x_from_limbs(point_ext + FP::X_LIMBS * i);
    HG_CUDA(cudaMemcpyAsync(pt.p, hpt.p, num_vars * sizeof(X), cudaMemcpyHostToDevice, s));
    const int lo = num_vars < 12 ? (int)num_vars : 12;
    const size_t nlo = (size_t)1 << lo, nhi = n >> lo;
    grow(eq, nlo + nhi);
    grow(out, n_tables);
    int blocks = (int)std::min<size_t>(nhi, (size_t)dev->sm_count * 2);
    grow(partials, (size_t)blocks * n_tables);
    grow(counters, n_tables);
    HG_CUDA(cudaMemsetAsync(counters.p, 0, n_tables * sizeof(unsigned), s));
    HG_K(dev, KC_EQ, (nlo + nhi) * sizeof(X), k_eq_split<FP><<<(unsigned)((nlo + nhi + HG_BLOCK - 1) / HG_BLOCK), HG_BLOCK, 0, s>>>(pt.p, (int)num_vars, lo, eq.p, eq.p + nlo));
    HG_K(dev, KC_DOT, n_tables * n * sizeof(B),
         k_dot_eq<FP, B><<<dim3(blocks, (unsigned)n_tables), HG_BLOCK, 0, s>>>((const B*)d_tables, stride, n, lo, eq.p, eq.p + nlo, partials.p, counters.p, out.p));
    X* ho = hpt.p + np;  // pinned
    HG_CUDA(cudaMemcpyAsync(ho, out.p, n_tables * sizeof(X), cudaMemcpyDeviceToHost, s));
    HG_CUDA(cudaStreamSynchronize(s));
    for (size_t i = 0; i < n_tables; i++) FP::x_to_limbs(ho[i], out_ext + FP::X_LIMBS * i);
}

// hg_bfv_witness_generate: scripts/circuit_sk.py:72-140 on the device (witness_gen.cuh). Small host inputs, device outputs in
// the library's representation.
template <class FP> void witness_generate(hg_ctx* ctx, size_t n, size_t K, const uint64_t* qis, const uint64_t* k0is, const uint64_t* r1b, const uint64_t* r2b,
                                          const int8_t* s, const int8_t* e, const int32_t* k1, const int64_t* a, void* d_s, void* d_e, void* d_k1, void* d_ais,
                                          void* d_r1is, void* d_r2is, void* d_ct0is) {
    typedef typename FP::B B;
    DeviceCtx* dev = &ctx->dev;
    FieldState<FP>& fs = typed<FP>(ctx);
    if (n < 2 || (n & (n - 1)) || K < 1 || K > 64) throw std::runtime_error("hg_bfv_witness_generate: n must be a power of two >= 2 and 1 <= K <= 64");
    cudaStream_t st = dev->stream;
    WitGenParams P;
    memset(&P, 0, sizeof P);
    P.n = (int)n; P.K = (int)K;
    for (size_t i = 0; i < K; i++) {
        if (qis[i] >= ((uint64_t)1 << 62) || qis[i] < 3) throw std::runtime_error("hg_bfv_witness_generate: modulus out of range");
        P.q[i] = (long long)qis[i]; P.k0[i] = (long long)k0is[i]; P.r1_bound[i] = (long long)r1b[i]; P.r2_bound[i] = (long long)r2b[i];
    }
    {   // p as canonical limbs: the limbs of -1 plus one
        B m1 = FP::b_sub(FP::b_zero(), FP::b_one());
        u64 l[4] = {0, 0, 0, 0};
        FP::b_to_limbs(m1, l);
        u64 c = 1;
        for (int q = 0; q < 4; q++) { const u64 v = l[q] + c; c = (v < l[q]) ? 1 : 0; P.p[q] = v; }
    }
    auto grow = [&](auto& buf, size_t need) { if (buf.n < need) { HG_CUDA(cudaStreamSynchronize(st)); buf.alloc(need); } };
    grow(fs.wg_s, n); grow(fs.wg_e, n); grow(fs.wg_k1, n); grow(fs.wg_a, K * n); grow(fs.wg_hat, K * 2 * n); grow(fs.wg_st, 1);
    HG_CUDA(cudaMemcpyAsync(fs.wg_s.p, s, n, cudaMemcpyHostToDevice, st));
    HG_CUDA(cudaMemcpyAsync(fs.wg_e.p, e, n, cudaMemcpyHostToDevice, st));
    HG_CUDA(cudaMemcpyAsync(fs.wg_k1.p, k1, n * sizeof(int), cudaMemcpyHostToDevice, st));
    HG_CUDA(cudaMemcpyAsync(fs.wg_a.p, a, K * n * sizeof(long long), cudaMemcpyHostToDevice, st));
    HG_CUDA(cudaMemsetAsync(fs.wg_st.p, 0, sizeof(WitGenStatus), st));
    const size_t N2 = 2 * n;
    HG_K(dev, KC_MISC, K * n * 8 + K * N2 * 16, k_wit_conv<<<dim3((unsigned)((N2 + HG_WIT_KT - 1) / HG_WIT_KT), (unsigned)K), HG_WIT_KT, 0, st>>>(fs.wg_s.p, fs.wg_a.p, (int)n, fs.wg_hat.p));
    constexpr int L = FP::B_LIMBS;
    HG_K(dev, KC_MISC, K * N2 * (16 + 3 * 8 * L),
         k_wit_finish<L><<<dim3((unsigned)((N2 + 255) / 256), (unsigned)K), 256, 0, st>>>(P, fs.wg_e.p, fs.wg_k1.p, fs.wg_a.p, fs.wg_hat.p, (u64*)d_ais, (u64*)d_r1is, (u64*)d_r2is,
                                                                                      (u64*)d_ct0is, fs.wg_st.p));
    HG_K(dev, KC_MISC, N2 * 3 * 8 * L, k_wit_small<L><<<(unsigned)((N2 + 255) / 256), 256, 0, st>>>(P, fs.wg_s.p, fs.wg_e.p, fs.wg_k1.p, (u64*)d_s, (u64*)d_e, (u64*)d_k1));
    if (FP::FIELD_ID == 1) {  // canonical limbs -> Montgomery form
        auto enc = [&](void* p, size_t cnt) { k_field_encode<FP><<<(unsigned)((cnt + 255) / 256), 256, 0, st>>>((B*)p, cnt, 0); HG_LAUNCH_CHECK(); };
        enc(d_s, N2); enc(d_e, N2); enc(d_k1, N2); enc(d_ais, K * N2); enc(d_r1is, K * N2); enc(d_r2is, K * n); enc(d_ct0is, K * N2);
    }
    WitGenStatus hs;
    HG_CUDA(cudaMemcpyAsync(&hs, fs.wg_st.p, sizeof hs, cudaMemcpyDeviceToHost, st));
    HG_CUDA(cudaStreamSynchronize(st));  // also keeps the caller's host arrays alive long enough
    if (hs.not_multiple_of_cyclo || hs.not_multiple_of_q || hs.r1_out_of_range || hs.r2_out_of_range)
        throw std::runtime_error("hg_bfv_witness_generate: assertion of circuit_sk.py failed: " + std::to_string(hs.not_multiple_of_cyclo) + " coefficients not a multiple of x^n+1, " +
                                 std::to_string(hs.not_multiple_of_q) + " not divisible by q_i, " + std::to_string(hs.r1_out_of_range) + " r1 out of range, " +
                                 std::to_string(hs.r2_out_of_range) + " r2 out of range");
}

// hg_field_selftest
template <class FP> void field_selftest(DeviceCtx* ctx, int op, const uint64_t* a_ext, const uint64_t* b_ext, size_t n, uint64_t* out_ext) {
    typedef typename FP::X X;
    std::vector<X> ha(n), hb(n), ho(n);
    for (size_t i = 0; i < n; i++) { ha[i] = FP::x_from_limbs(a_ext + i * FP::X_LIMBS); hb[i] = FP::x_from_limbs(b_ext + i * FP::X_LIMBS); }
    DevBuf<X> a, b, o;
    a.alloc(n); b.alloc(n); o.alloc(n);
    // stream-ordered copies: a blocking cudaMemcpy from pageable memory runs on the legacy stream, which a non-blocking stream does not wait for
    HG_CUDA(cudaMemcpyAsync(a.p, ha.data(), n * sizeof(X), cudaMemcpyHostToDevice, ctx->stream));
    HG_CUDA(cudaMemcpyAsync(b.p, hb.data(), n * sizeof(X), cudaMemcpyHostToDevice, ctx->stream));
    k_selftest<FP><<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(op, a.p, b.p, n, o.p);
    HG_LAUNCH_CHECK();
    HG_CUDA(cudaMemcpyAsync(ho.data(), o.p, n * sizeof(X), cudaMemcpyDeviceToHost, ctx->stream));
    HG_CUDA(cudaStreamSynchronize(ctx->stream));
    for (size_t i = 0; i < n; i++) FP::x_to_limbs(ho[i], out_ext + i * FP::X_LIMBS);
}

extern "C" {

const char* hg_last_error(void) { return g_err.c_str(); }
int hg_version(void) { return 2; }

int hg_ctx_create(int device, int field_id, hg_ctx** out) {
    HG_TRY({
        int n = 0;
        HG_CUDA(cudaGetDeviceCount(&n));
        if (device < 0 || device >= n) throw std::runtime_error("no such CUDA device");
        HG_CUDA(cudaSetDevice(device));
        struct CtxDeleter { void operator()(hg_ctx* p) const { hg_ctx_destroy(p); } };  // a failing call below must not leak the streams / events made before it
        std::unique_ptr<hg_ctx, CtxDeleter> c(new hg_ctx());
        with_field(field_id, [&](auto fp) { c->state.template emplace<FieldState<decltype(fp)>>(); });
        c->dev.device = device;
        c->field_id = field_id;
        HG_CUDA(cudaStreamCreateWithFlags(&c->dev.stream, cudaStreamNonBlocking));
        {   // second stream for work that is independent of the Lasso node (the generic layer sumchecks): higher priority so
            // that its short kernels are dispatched as soon as blocks of the long streaming kernels retire
            int lo = 0, hi = 0;
            HG_CUDA(cudaDeviceGetStreamPriorityRange(&lo, &hi));
            HG_CUDA(cudaStreamCreateWithPriority(&c->dev.stream2, cudaStreamNonBlocking, hi));
            HG_CUDA(cudaEventCreateWithFlags(&c->dev.ev_fork, cudaEventDisableTiming));
            HG_CUDA(cudaEventCreateWithFlags(&c->dev.ev_join, cudaEventDisableTiming));
            HG_CUDA(cudaStreamCreateWithFlags(&c->dev.stream3, cudaStreamNonBlocking));
            HG_CUDA(cudaEventCreateWithFlags(&c->dev.ev_fork3, cudaEventDisableTiming));
            HG_CUDA(cudaEventCreateWithFlags(&c->dev.ev_join3, cudaEventDisableTiming));
            HG_CUDA(cudaEventCreateWithFlags(&c->dev.ev_coll, cudaEventDisableTiming));
        }
        HG_CUDA(cudaDeviceGetAttribute(&c->dev.sm_count, cudaDevAttrMultiProcessorCount, device));
        *out = c.release();
    })
}
void hg_ctx_destroy(hg_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->dev.device);
    ctx->state.emplace<std::monostate>();  // the NTT engine and work buffers go while the streams still exist
    if (ctx->dev.ev_fork) cudaEventDestroy(ctx->dev.ev_fork);
    if (ctx->dev.ev_join) cudaEventDestroy(ctx->dev.ev_join);
    if (ctx->dev.ev_fork3) cudaEventDestroy(ctx->dev.ev_fork3);
    if (ctx->dev.ev_join3) cudaEventDestroy(ctx->dev.ev_join3);
    if (ctx->dev.ev_coll) cudaEventDestroy(ctx->dev.ev_coll);
    if (ctx->dev.stream3) cudaStreamDestroy(ctx->dev.stream3);
    if (ctx->dev.stream2) cudaStreamDestroy(ctx->dev.stream2);
    if (ctx->dev.stream) cudaStreamDestroy(ctx->dev.stream);
    delete ctx;
}
int hg_ctx_set_option(hg_ctx* ctx, int option, int value) {
    HG_TRY({
        if (option == HG_OPT_A3_WIRE) ctx->wire.a3_wire = value;
        else if (option == HG_OPT_A3_H1) ctx->wire.a3_h1 = value;
        else if (option == HG_OPT_A5_ASCENDING) ctx->wire.a5_ascending = value;
        else if (option == HG_OPT_TWO_STREAMS) ctx->dev.two_streams = value != 0;
        else throw std::runtime_error("unknown option");
    })
}
int hg_ctx_synchronize(hg_ctx* ctx) { HG_TRY({ HG_CUDA(cudaSetDevice(ctx->dev.device)); HG_CUDA(cudaStreamSynchronize(ctx->dev.stream)); }) }
uint64_t hg_ctx_launch_count(hg_ctx* ctx) { return ctx->dev.launches; }
int hg_ctx_profile(hg_ctx* ctx, int enable) {
    HG_TRY({
        HG_CUDA(cudaSetDevice(ctx->dev.device));
        ctx->dev.profile_collect();
        if (enable) ctx->dev.profile_reset();
        ctx->dev.profile = enable != 0;
    })
}
int hg_ctx_profile_read(hg_ctx* ctx, int kernel_class, uint64_t* launches, double* ms, uint64_t* algorithmic_bytes) {
    HG_TRY({
        if (kernel_class < 0 || kernel_class >= KC_COUNT) throw std::runtime_error("no such kernel class");
        HG_CUDA(cudaSetDevice(ctx->dev.device));
        ctx->dev.profile_collect();
        *launches = ctx->dev.cls_launches[kernel_class];
        *ms = ctx->dev.cls_ms[kernel_class];
        *algorithmic_bytes = ctx->dev.cls_bytes[kernel_class];
    })
}
int hg_kernel_class_count(void) { return KC_COUNT; }
const char* hg_kernel_class_name(int kernel_class) { return kernel_class_name(kernel_class); }
void* hg_ctx_stream(hg_ctx* ctx) { return (void*)ctx->dev.stream; }
size_t hg_field_base_bytes(int field_id) { return field_id == HG_FIELD_BN254 ? sizeof(FrField::B) : sizeof(GlField::B); }  // Goldilocks' for an unknown id

int hg_buf_alloc(hg_ctx* ctx, size_t bytes, hg_buf** out) {
    HG_TRY({
        HG_CUDA(cudaSetDevice(ctx->dev.device));
        std::unique_ptr<hg_buf> b(new hg_buf());
        HG_CUDA(cudaMalloc(&b->p, bytes ? bytes : 1));
        b->bytes = bytes;
        b->device = ctx->dev.device;
        *out = b.release();
    })
}
int hg_buf_upload(hg_ctx* ctx, hg_buf* buf, size_t offset, const void* host, size_t bytes) {
    HG_TRY({
        if (offset + bytes > buf->bytes) throw std::runtime_error("hg_buf_upload: out of range");
        HG_CUDA(cudaSetDevice(ctx->dev.device));
        HG_CUDA(cudaMemcpyAsync((char*)buf->p + offset, host, bytes, cudaMemcpyHostToDevice, ctx->dev.stream));
        HG_CUDA(cudaStreamSynchronize(ctx->dev.stream));
    })
}
int hg_buf_upload_async(hg_ctx* ctx, hg_buf* buf, size_t offset, const void* host, size_t bytes) {
    HG_TRY({
        if (offset + bytes > buf->bytes) throw std::runtime_error("hg_buf_upload_async: out of range");
        HG_CUDA(cudaSetDevice(ctx->dev.device));
        HG_CUDA(cudaMemcpyAsync((char*)buf->p + offset, host, bytes, cudaMemcpyHostToDevice, ctx->dev.stream));
    })
}
int hg_buf_download(hg_ctx* ctx, const hg_buf* buf, size_t offset, void* host, size_t bytes) {
    HG_TRY({
        if (offset + bytes > buf->bytes) throw std::runtime_error("hg_buf_download: out of range");
        HG_CUDA(cudaSetDevice(ctx->dev.device));
        HG_CUDA(cudaMemcpyAsync(host, (const char*)buf->p + offset, bytes, cudaMemcpyDeviceToHost, ctx->dev.stream));
        HG_CUDA(cudaStreamSynchronize(ctx->dev.stream));
    })
}
int hg_device_download(hg_ctx* ctx, const void* d_ptr, void* host, size_t bytes) {
    HG_TRY({
        if (!d_ptr || !host) throw std::runtime_error("hg_device_download: NULL pointer");
        HG_CUDA(cudaSetDevice(ctx->dev.device));
        HG_CUDA(cudaMemcpyAsync(host, d_ptr, bytes, cudaMemcpyDeviceToHost, ctx->dev.stream));
        HG_CUDA(cudaStreamSynchronize(ctx->dev.stream));
    })
}
void* hg_buf_device_ptr(hg_buf* buf) { return buf->p; }
size_t hg_buf_size(const hg_buf* buf) { return buf->bytes; }
void hg_buf_free(hg_buf* buf) {
    if (!buf) return;
    cudaSetDevice(buf->device);
    cudaFree(buf->p);
    delete buf;
}
// device tables hold the library's internal representation: canonical u64 for Goldilocks, 4x64 Montgomery for BN254.
// hg_field_encode converts n base elements uploaded as canonical little-endian limbs in place; hg_field_decode goes back.
static void field_encode(hg_ctx* ctx, void* d, size_t n, bool decode) {
    HG_CUDA(cudaSetDevice(ctx->dev.device));
    with_field(ctx->field_id, [&](auto fp) {
        typedef decltype(fp) FP;
        if (FP::FIELD_ID != 1 || !n) return;
        k_field_encode<FP><<<(unsigned)((n + 255) / 256), 256, 0, ctx->dev.stream>>>((typename FP::B*)d, n, decode ? 1 : 0);
        HG_LAUNCH_CHECK();
        HG_CUDA(cudaStreamSynchronize(ctx->dev.stream));
    });
}
int hg_field_encode(hg_ctx* ctx, void* d_data, size_t n) { HG_TRY({ field_encode(ctx, d_data, n, false); }) }
int hg_field_decode(hg_ctx* ctx, void* d_data, size_t n) { HG_TRY({ field_encode(ctx, d_data, n, true); }) }

// ---- transcript
int hg_transcript_new(int field_id, hg_transcript** out) { HG_TRY({ *out = new_transcript(field_id); }) }
int hg_transcript_from_proof(int field_id, const uint8_t* proof, size_t len, hg_transcript** out) { HG_TRY({ *out = new_transcript(field_id, proof, len); }) }
int hg_transcript_from_callbacks(int field_id, void* user, hg_squeeze_fn squeeze, hg_write_fn write, hg_read_fn read, int message_independent,
                                 hg_transcript** out) {
    HG_TRY({
        if (!out) throw std::runtime_error("hg_transcript_from_callbacks: out is NULL");
        if (!squeeze) throw std::runtime_error("hg_transcript_from_callbacks: a squeeze callback is required");
        TranscriptHooks h;
        h.user = user; h.squeeze = squeeze; h.write = write; h.read = read; h.message_independent = message_independent != 0;
        *out = new_transcript(field_id, h);
    })
}
void hg_transcript_free(hg_transcript* t) { delete t; }
int hg_transcript_squeeze_challenges(hg_transcript* t, size_t n, uint64_t* out_ext) {
    HG_TRY({
        std::visit([&](auto& tr) {
            typedef field_t<decltype(tr)> FP;
            for (size_t i = 0; i < n; i++) FP::x_to_limbs(tr.squeeze_challenge(), out_ext + i * FP::X_LIMBS);
        }, t->t);
    })
}
int hg_transcript_squeeze_challenge(hg_transcript* t, uint64_t* out_ext) { return hg_transcript_squeeze_challenges(t, 1, out_ext); }
int hg_transcript_write_felt_ext(hg_transcript* t, const uint64_t* ext) {
    HG_TRY({ std::visit([&](auto& tr) { tr.write_felt_ext(field_t<decltype(tr)>::x_from_limbs(ext)); }, t->t); })
}
int hg_transcript_read_felt_ext(hg_transcript* t, uint64_t* out_ext) {
    HG_TRY({ std::visit([&](auto& tr) { field_t<decltype(tr)>::x_to_limbs(tr.read_felt_ext(), out_ext); }, t->t); })
}
size_t hg_transcript_proof_len(const hg_transcript* t) { return proof_bytes(t).size(); }
int hg_transcript_proof_copy(const hg_transcript* t, uint8_t* out, size_t cap) {
    HG_TRY({
        auto& p = proof_bytes(t);
        if (p.size() > cap) throw std::runtime_error("hg_transcript_proof_copy: buffer too small");
        memcpy(out, p.data(), p.size());
    })
}
int hg_transcript_append_bytes(hg_transcript* t, const uint8_t* bytes, size_t n) {
    HG_TRY({ std::visit([&](auto& tr) { tr.append_raw(bytes, n); }, t->t); })
}
size_t hg_transcript_num_squeezed(const hg_transcript* t) { return std::visit([](auto& tr) { return tr.num_base_squeezed(); }, t->t); }

// ---- preprocessing
int hg_lasso_preprocess(const uint64_t* bounds, size_t n_bounds, size_t C, size_t M, hg_lasso_pp** out) {
    HG_TRY({
        if (M < 2 || (M & (M - 1))) throw std::runtime_error("M must be a power of two >= 2");
        std::vector<std::shared_ptr<LookupType>> lk;
        for (size_t i = 0; i < n_bounds; i++) lk.push_back(std::make_shared<RangeLookup>(bounds[i]));
        std::unique_ptr<hg_lasso_pp> h(new hg_lasso_pp());
        h->pp = LassoPreprocessing::preprocess(lk, C, M);
        for (auto& l : h->pp.lookups) h->lookup_bounds.push_back(static_cast<RangeLookup*>(l.get())->bound());
        *out = h.release();
    })
}
int hg_lasso_preprocess_lookups(const hg_lookup_desc* lookups, size_t n_lookups, size_t C, size_t M, hg_lasso_pp** out) {
    HG_TRY({
        if (M < 2 || (M & (M - 1))) throw std::runtime_error("M must be a power of two >= 2");
        if (!lookups || !out || n_lookups < 1) throw std::runtime_error("hg_lasso_preprocess_lookups: NULL argument or no lookups");
        if (C < 1 || C > (size_t)HG_MAX_C) throw std::runtime_error("hg_lasso_preprocess_lookups: C out of range");
        const unsigned log2M = ilog2u(M);
        std::map<std::string, std::shared_ptr<LassoSubtable>> tables;  // one object per subtable id: the same id must mean the same table
        std::vector<std::shared_ptr<LookupType>> lk;
        for (size_t i = 0; i < n_lookups; i++) {
            const hg_lookup_desc& d = lookups[i];
            if (!d.lookup_id || !d.subtable_ids || !d.tables || !d.dimension_masks || !d.chunk_bits || d.n_subtables < 1 || d.n_chunk_bits < 1 || d.n_chunk_bits > C)
                throw std::runtime_error("hg_lasso_preprocess_lookups: malformed descriptor " + std::to_string(i));
            std::vector<std::pair<std::shared_ptr<LassoSubtable>, SubtableIndices>> sts;
            uint64_t covered = 0;
            for (size_t q = 0; q < d.n_subtables; q++) {
                if (!d.subtable_ids[q] || !d.tables[q]) throw std::runtime_error("hg_lasso_preprocess_lookups: NULL subtable in descriptor " + std::to_string(i));
                if (d.dimension_masks[q] == 0 || (d.dimension_masks[q] >> d.n_chunk_bits)) throw std::runtime_error("hg_lasso_preprocess_lookups: a subtable must serve dimensions below the chunk count");
                const std::string id = d.subtable_ids[q];
                std::vector<uint64_t> t(d.tables[q], d.tables[q] + M);
                auto it = tables.find(id);
                if (it == tables.end()) it = tables.emplace(id, std::make_shared<TableSubtable>(id, t)).first;
                else if (it->second->materialize(M) != t) throw std::runtime_error("hg_lasso_preprocess_lookups: subtable id '" + id + "' is used for two different tables");
                sts.push_back({it->second, SubtableIndices::from_mask(d.dimension_masks[q])});
                covered |= d.dimension_masks[q];
            }
            if (covered != (((uint64_t)1 << d.n_chunk_bits) - 1)) throw std::runtime_error("hg_lasso_preprocess_lookups: every chunk of lookup '" + std::string(d.lookup_id) + "' needs a subtable");
            std::vector<unsigned> cb(d.chunk_bits, d.chunk_bits + d.n_chunk_bits);
            for (unsigned b : cb) if (b < 1 || b > log2M) throw std::runtime_error("hg_lasso_preprocess_lookups: chunk_bits must be in 1..=log2(M)");
            lk.push_back(std::make_shared<TableLookup>(d.lookup_id, sts, cb, d.combine_weight));
        }
        std::unique_ptr<hg_lasso_pp> h(new hg_lasso_pp());
        h->pp = LassoPreprocessing::preprocess(lk, C, M);
        *out = h.release();
    })
}
int hg_lasso_pp_lookup_index_by_id(const hg_lasso_pp* pp, const char* lookup_id) {
    if (!pp || !lookup_id) return -1;
    auto it = pp->pp.lookup_id_to_index.find(lookup_id);
    return it == pp->pp.lookup_id_to_index.end() ? -1 : (int)it->second;
}
int hg_lasso_node_new_ids(hg_ctx* ctx, const hg_lasso_pp* pp, size_t num_vars, const char* const* seg_lookup_ids, const uint64_t* seg_lens, size_t n_segs,
                          hg_lasso_node** out) {
    HG_TRY({
        HG_CUDA(cudaSetDevice(ctx->dev.device));
        if (num_vars < 1 || num_vars > 30) throw std::runtime_error("num_vars out of range");
        if (!seg_lookup_ids || !seg_lens || !out) throw std::runtime_error("hg_lasso_node_new_ids: NULL argument");
        std::vector<uint8_t> rows;
        for (size_t s = 0; s < n_segs; s++) {
            const int li = hg_lasso_pp_lookup_index_by_id(pp, seg_lookup_ids[s]);
            if (li < 0) throw std::runtime_error("lookup id " + std::string(seg_lookup_ids[s] ? seg_lookup_ids[s] : "(null)") + " not in preprocessing");
            rows.insert(rows.end(), seg_lens[s], (uint8_t)li);
        }
        *out = new_lasso_node(ctx, pp, num_vars, rows);
    })
}
void hg_lasso_pp_free(hg_lasso_pp* pp) { delete pp; }
size_t hg_lasso_pp_num_lookups(const hg_lasso_pp* pp) { return pp->pp.lookups.size(); }
size_t hg_lasso_pp_num_subtables(const hg_lasso_pp* pp) { return pp->pp.subtables_by_idx.size(); }
size_t hg_lasso_pp_num_memories(const hg_lasso_pp* pp) { return pp->pp.num_memories; }
int hg_lasso_pp_lookup_index(const hg_lasso_pp* pp, uint64_t bound) {
    auto it = pp->pp.lookup_id_to_index.find(RangeLookup::id_for(bound));
    return it == pp->pp.lookup_id_to_index.end() ? -1 : (int)it->second;
}
int hg_lasso_pp_memory_maps(const hg_lasso_pp* pp, uint32_t* mem_to_subtable, uint32_t* mem_to_dimension) {
    HG_TRY({
        for (size_t i = 0; i < pp->pp.num_memories; i++) {
            if (mem_to_subtable) mem_to_subtable[i] = (uint32_t)pp->pp.memory_to_subtable_index[i];
            if (mem_to_dimension) mem_to_dimension[i] = (uint32_t)pp->pp.memory_to_dimension_index[i];
        }
    })
}
int hg_lasso_pp_subtable_id(const hg_lasso_pp* pp, size_t idx, char* out, size_t cap) {
    HG_TRY({
        if (idx >= pp->pp.subtables_by_idx.size()) throw std::runtime_error("subtable index out of range");
        std::string id = pp->pp.subtables_by_idx[idx]->subtable_id();
        if (id.size() + 1 > cap) throw std::runtime_error("buffer too small");
        memcpy(out, id.c_str(), id.size() + 1);
    })
}

// ---- node
int hg_lasso_node_new(hg_ctx* ctx, const hg_lasso_pp* pp, size_t num_vars, const uint64_t* seg_bounds, const uint64_t* seg_lens, size_t n_segs,
                      hg_lasso_node** out) {
    HG_TRY({
        HG_CUDA(cudaSetDevice(ctx->dev.device));
        if (num_vars < 1 || num_vars > 30) throw std::runtime_error("num_vars out of range");
        std::vector<uint8_t> rows;
        for (size_t s = 0; s < n_segs; s++) {
            int li = hg_lasso_pp_lookup_index(pp, seg_bounds[s]);
            if (li < 0) throw std::runtime_error("lookup id " + RangeLookup::id_for(seg_bounds[s]) + " not in preprocessing");
            rows.insert(rows.end(), seg_lens[s], (uint8_t)li);
        }
        *out = new_lasso_node(ctx, pp, num_vars, rows);
    })
}
void hg_lasso_node_free(hg_lasso_node* node) {
    if (!node) return;
    cudaSetDevice(node->ctx->dev.device);
    delete node;
}
size_t hg_lasso_node_log2_input_size(const hg_lasso_node* node) { return node->log2_input_size; }
size_t hg_lasso_node_device_bytes(const hg_lasso_node* node) { return std::visit([](auto& n) { return n.device_bytes(); }, node->node); }
size_t hg_lasso_node_num_chunks(const hg_lasso_node* node) { return std::visit([](auto& n) { return n.chunk_dims().size(); }, node->node); }
void hg_lasso_node_timing(const hg_lasso_node* node, double* out_us4) {
    const double* t = std::visit([](auto& n) { return n.timing(); }, node->node);
    for (int i = 0; i < 4; i++) out_us4[i] = t[i];
}

int hg_lasso_node_prove(hg_lasso_node* node, const void* inputs, size_t n_inputs, int inputs_on_device, hg_transcript* t, int mode,
                        uint64_t* out_point, uint64_t* out_value) {
    HG_TRY({
        hg_ctx* ctx = node->ctx;
        HG_CUDA(cudaSetDevice(ctx->dev.device));
        std::visit([&](auto& n) {
            typedef field_t<decltype(n)> FP;
            Keccak256Transcript<FP>& tr = typed<FP>(t);
            std::vector<typename FP::X> pt;
            typename FP::X val;
            n.prove(stage<FP>(node, inputs, n_inputs, inputs_on_device != 0), n_inputs, tr, mode == HG_MODE_INTERACTIVE ? kModeInteractive : kModePrefetch, ctx->wire, &pt, &val);
            claim_to_limbs<FP>(pt, val, out_point, out_value);
        }, node->node);
    })
}
size_t hg_lasso_node_shard_words(const hg_lasso_node* node) {
    return std::visit([](auto& n) { return n.shard_message_count() * XW<field_t<decltype(n)>>; }, node->node);
}
// the partial message buffer goes to host or device memory alike; the host-words entry point waits for it
int hg_lasso_node_prove_shard(hg_lasso_node* node, const void* inputs, size_t n_inputs, int inputs_on_device, hg_transcript* t, int rank, int world,
                              uint64_t* out_words, size_t cap_words, size_t* n_words) {
    const int rc = hg_lasso_node_prove_shard_dev(node, inputs, n_inputs, inputs_on_device, t, rank, world, out_words, cap_words, n_words);
    return rc ? rc : hg_ctx_synchronize(node->ctx);
}
int hg_lasso_node_prove_shard_dev(hg_lasso_node* node, const void* inputs, size_t n_inputs, int inputs_on_device, hg_transcript* t, int rank, int world,
                                  void* d_out_words, size_t cap_words, size_t* n_words) {
    HG_TRY({
        HG_CUDA(cudaSetDevice(node->ctx->dev.device));
        if (!d_out_words || !n_words) throw std::runtime_error("hg_lasso_node_prove_shard_dev: NULL output");
        std::visit([&](auto& n) {
            typedef field_t<decltype(n)> FP;
            Keccak256Transcript<FP>& tr = typed<FP>(t);
            *n_words = XW<FP> * n.prove_shard(stage<FP>(node, inputs, n_inputs, inputs_on_device != 0), n_inputs, tr, node->ctx->wire, rank, world,
                                              (typename FP::X*)d_out_words, cap_words / XW<FP>);
        }, node->node);
    })
}
// the merged buffer may be host or device memory
int hg_lasso_node_emit_shard(hg_lasso_node* node, const uint64_t* merged_words, size_t n_words, uint64_t* out_point, uint64_t* out_value) {
    return hg_lasso_node_emit_shard_dev(node, merged_words, n_words, out_point, out_value);
}
int hg_lasso_node_emit_shard_dev(hg_lasso_node* node, const void* d_merged_words, size_t n_words, uint64_t* out_point, uint64_t* out_value) {
    HG_TRY({
        HG_CUDA(cudaSetDevice(node->ctx->dev.device));
        std::visit([&](auto& n) {
            typedef field_t<decltype(n)> FP;
            if (n_words % XW<FP>) throw std::runtime_error("emit_shard: truncated message buffer");
            std::vector<typename FP::X> pt;
            typename FP::X val;
            n.emit_shard((const typename FP::X*)d_merged_words, n_words / XW<FP>, &pt, &val);
            claim_to_limbs<FP>(pt, val, out_point, out_value);
        }, node->node);
    })
}
int hg_shard_merge_device(hg_ctx* ctx, const void* d_parts_words, int world, size_t n_words, void* d_acc_words) {
    HG_TRY({
        HG_CUDA(cudaSetDevice(ctx->dev.device));
        with_field(ctx->field_id, [&](auto fp) {
            typedef decltype(fp) FP;
            typedef typename FP::X X;
            if (n_words % XW<FP> || world < 1) throw std::runtime_error("hg_shard_merge_device: bad arguments");
            const size_t n = n_words / XW<FP>;
            if (!n) return;
            HG_K(&ctx->dev, KC_MISC, 0, k_shard_merge<FP><<<(unsigned)((n + 255) / 256), 256, 0, ctx->dev.stream>>>((const X*)d_parts_words, world, n, (X*)d_acc_words));
        });
    })
}
size_t hg_gkr_shard_words(hg_circuit* c) {
    try {
        if (!c->ctx) return 0;
        return with_kind<GkrCircuitDev>(c, [](auto& dc) { return dc.shard_message_count() * XW<field_t<decltype(dc)>>; });
    } catch (...) { cudaGetLastError(); return 0; }
}
int hg_gkr_prove_shard_dev(hg_circuit* c, size_t n_output_claims, const size_t* point_lens, const uint64_t* points_ext, const uint64_t* values_ext, hg_transcript* t,
                           int rank, int world, void* d_out_words, size_t cap_words, size_t* n_words) {
    HG_TRY({
        circuit_use_device(c);
        if (!d_out_words || !n_words) throw std::runtime_error("hg_gkr_prove_shard_dev: NULL output");
        with_kind<GkrCircuitDev>(c, [&](auto& dc) {
            typedef field_t<decltype(dc)> FP;
            Keccak256Transcript<FP>& tr = typed<FP>(t);
            auto oc = claims_from_limbs<FP, typename GkrCircuitDev<FP>::InputClaim>(n_output_claims, point_lens, points_ext, values_ext);
            *n_words = XW<FP> * dc.prove_shard_dev(tr, c->ctx->wire, oc, rank, world, (typename FP::X*)d_out_words, cap_words / XW<FP>);
        });
    })
}
int hg_gkr_emit_shard_dev(hg_circuit* c, const void* d_merged_words, size_t n_words) {
    HG_TRY({
        circuit_use_device(c);
        with_kind<GkrCircuitDev>(c, [&](auto& dc) {
            typedef field_t<decltype(dc)> FP;
            if (n_words % XW<FP>) throw std::runtime_error("emit_shard: truncated message buffer");
            set_input_claims<FP>(c, dc.emit_shard_dev((const typename FP::X*)d_merged_words, n_words / XW<FP>));
        });
    })
}
int hg_gkr_emit_shard_part_dev(hg_circuit* c, const void* d_merged_words, size_t n_words, int part, int nparts, uint8_t* out_bytes, size_t cap, size_t* out_len) {
    HG_TRY({
        circuit_use_device(c);
        if (!out_bytes || !out_len) throw std::runtime_error("hg_gkr_emit_shard_part_dev: NULL output");
        std::vector<uint8_t> bytes;
        with_kind<GkrCircuitDev>(c, [&](auto& dc) {
            typedef field_t<decltype(dc)> FP;
            if (n_words % XW<FP>) throw std::runtime_error("emit_shard: truncated message buffer");
            set_input_claims<FP>(c, dc.emit_shard_part_dev((const typename FP::X*)d_merged_words, n_words / XW<FP>, part, nparts, bytes));
        });
        if (bytes.size() > cap) throw std::runtime_error("hg_gkr_emit_shard_part_dev: output buffer too small");
        if (!bytes.empty()) memcpy(out_bytes, bytes.data(), bytes.size());
        *out_len = bytes.size();
    })
}
int hg_lasso_node_verify(const hg_lasso_pp* pp, size_t num_vars, hg_transcript* t, const int* options3, uint64_t* out_point, uint64_t* out_value) {
    HG_TRY({
        const WireOptions wo = wire_options(options3);
        std::visit([&](auto& tr) {
            typedef field_t<decltype(tr)> FP;
            LassoVerifier<FP> v(pp->pp, (int)num_vars, wo);
            std::vector<typename FP::X> r;
            typename FP::X sum;
            v.verify(tr, &r, &sum);
            claim_to_limbs<FP>(r, sum, out_point, out_value);
        }, t->t);
    })
}
int hg_shard_merge(int field, uint64_t* acc_words, const uint64_t* part_words, size_t n_words) {
    HG_TRY({
        with_field(field, [&](auto fp) {
            typedef decltype(fp) FP;
            typedef typename FP::X X;
            if (n_words % XW<FP>) throw std::runtime_error("shard_merge: truncated message buffer");
            X* a = (X*)acc_words;
            const X* b = (const X*)part_words;
            for (size_t i = 0; i < n_words / XW<FP>; i++) a[i] = FP::x_add(a[i], b[i]);
        });
    })
}
int hg_lasso_node_download_polys(hg_lasso_node* node, uint16_t* dims, uint32_t* read_cts, uint32_t* final_cts, uint64_t* e_polys) {
    HG_TRY({
        HG_CUDA(cudaSetDevice(node->ctx->dev.device));
        std::visit([&](auto& n) {
            typedef field_t<decltype(n)> FP;
            std::vector<u16> d; std::vector<u32> r, f; std::vector<typename FP::B> e;
            n.download_polys(dims ? &d : nullptr, read_cts ? &r : nullptr, final_cts ? &f : nullptr, e_polys ? &e : nullptr);
            if (dims) memcpy(dims, d.data(), d.size() * sizeof(u16));
            if (read_cts) memcpy(read_cts, r.data(), r.size() * sizeof(u32));
            if (final_cts) memcpy(final_cts, f.data(), f.size() * sizeof(u32));
            if (e_polys) for (size_t i = 0; i < e.size(); i++) FP::b_to_limbs(e[i], e_polys + i * FP::B_LIMBS);
        }, node->node);
    })
}

// ---- generic sumcheck / MLE / NTT / forward evaluation
int hg_sumcheck_prove(hg_ctx* ctx, int arity, size_t n_terms, size_t num_vars, const uint64_t* coeffs_ext, const void* d_tables,
                      const uint64_t* claim_ext, hg_transcript* t, int mode, uint64_t* out_point, uint64_t* out_evals) {
    HG_TRY({
        HG_CUDA(cudaSetDevice(ctx->dev.device));
        with_field(ctx->field_id, [&](auto fp) { sumcheck_prove<decltype(fp)>(ctx, arity, n_terms, num_vars, coeffs_ext, d_tables, claim_ext, t, mode, out_point, out_evals); });
    })
}
int hg_mle_eval_batch(hg_ctx* ctx, const void* d_tables, size_t n_tables, size_t stride, size_t num_vars, const uint64_t* point_ext,
                      uint64_t* out_ext) {
    HG_TRY({
        HG_CUDA(cudaSetDevice(ctx->dev.device));
        with_field(ctx->field_id, [&](auto fp) { mle_eval_batch<decltype(fp)>(ctx, d_tables, n_tables, stride, num_vars, point_ext, out_ext); });
    })
}
int hg_ntt(hg_ctx* ctx, void* d_data, size_t log_n, int inverse, size_t batch) {
    HG_TRY({
        HG_CUDA(cudaSetDevice(ctx->dev.device));
        with_field(ctx->field_id, [&](auto fp) {
            typedef decltype(fp) FP;
            typed<FP>(ctx).eng(&ctx->dev)->run((typename FP::B*)d_data, (int)log_n, inverse != 0, batch);
        });
    })
}
int hg_bfv_configure(hg_circuit* c, size_t log2_size, size_t K, const uint64_t* qis, const uint64_t* k0is, const uint64_t* r1_bounds, const uint64_t* r2_bounds,
                     uint64_t s_bound, uint64_t e_bound, uint64_t k1_bound, hg_lasso_node* lasso_node, const hg_lasso_pp* lasso_pp, size_t lasso_num_vars,
                     int* out_ids6) {
    HG_TRY({
        if (!c || !qis || !k0is || !r1_bounds || !r2_bounds || K < 1 || K > 4096) throw std::runtime_error("hg_bfv_configure: bad arguments");
        if (c->ctx) circuit_use_device(c);
        if (c->ctx && !lasso_node) throw std::runtime_error("hg_bfv_configure: a device circuit needs the Lasso node (hg_lasso_node_new)");
        if (!c->ctx && !lasso_pp) throw std::runtime_error("hg_bfv_configure: a host-only circuit needs the Lasso preprocessing and num_vars");
        BfvCircuitParams P;
        P.log2_size = log2_size; P.K = K; P.s_bound = s_bound; P.e_bound = e_bound; P.k1_bound = k1_bound;
        P.qis.assign(qis, qis + K); P.k0is.assign(k0is, k0is + K); P.r1_bounds.assign(r1_bounds, r1_bounds + K); P.r2_bounds.assign(r2_bounds, r2_bounds + K);
        const BfvCircuitIds id = std::visit([&](auto& k) {
            typedef std::remove_reference_t<decltype(k)> Ckt;
            typedef field_t<Ckt> FP;
            std::function<int()> ins;
            if constexpr (std::is_same_v<Ckt, GkrCircuitDev<FP>>) ins = [&k, n = &typed<FP>(lasso_node)]() { return k.insert_lasso(n); };
            else ins = [&]() { return k.insert_lasso(lasso_pp->pp, (int)lasso_num_vars); };
            return bfv_configure<FP::B_LIMBS>(k, P, ins);
        }, c->c);
        if (out_ids6) { out_ids6[0] = id.s; out_ids6[1] = id.e; out_ids6[2] = id.k1; out_ids6[3] = id.lasso_in; out_ids6[4] = id.lasso; out_ids6[5] = id.sum; }
    })
}

// ---- circuit-level API: Circuit::{insert, connect, evaluate} + prove_gkr
int hg_circuit_new(hg_ctx* ctx, hg_circuit** out) {
    HG_TRY({
        HG_CUDA(cudaSetDevice(ctx->dev.device));
        *out = with_field(ctx->field_id, [&](auto fp) {
            typedef decltype(fp) FP;
            return new hg_circuit(ctx, ctx->field_id, std::in_place_type<GkrCircuitDev<FP>>, &ctx->dev, typed<FP>(ctx).eng(&ctx->dev));
        });
    })
}
int hg_circuit_new_host(int field_id, hg_circuit** out) {
    HG_TRY({
        if (!out) throw std::runtime_error("hg_circuit_new_host: out is NULL");
        *out = with_field(field_id, [&](auto fp) { return new hg_circuit(nullptr, field_id, std::in_place_type<GkrVerifierHost<decltype(fp)>>); });
    })
}
int hg_circuit_insert_lasso_host(hg_circuit* c, const hg_lasso_pp* pp, size_t num_vars, int* out_id) {
    HG_TRY({
        if (c->ctx) throw std::runtime_error("hg_circuit_insert_lasso_host needs a host-only circuit (hg_circuit_new_host)");
        with_kind<GkrVerifierHost>(c, [&](auto& v) { *out_id = v.insert_lasso(pp->pp, (int)num_vars); });
    })
}
int hg_gkr_verify(hg_circuit* c, size_t n_output_claims, const size_t* point_lens, const uint64_t* points_ext, const uint64_t* values_ext, hg_transcript* t,
                  const int* options3) {
    HG_TRY({
        const WireOptions wo = wire_options(options3);
        if (c->ctx) throw std::runtime_error("hg_gkr_verify needs a host-only circuit description (hg_circuit_new_host)");
        with_kind<GkrVerifierHost>(c, [&](auto& v) {
            typedef field_t<decltype(v)> FP;
            Keccak256Transcript<FP>& tr = typed<FP>(t);
            auto oc = claims_from_limbs<FP, typename GkrVerifierHost<FP>::Claim>(n_output_claims, point_lens, points_ext, values_ext);
            set_input_claims<FP>(c, v.verify(tr, wo, oc));
        });
    })
}
int hg_bfv_witness_generate(hg_ctx* ctx, size_t n, size_t K, const uint64_t* qis, const uint64_t* k0is, const uint64_t* r1_bounds, const uint64_t* r2_bounds,
                            const int8_t* s, const int8_t* e, const int32_t* k1, const int64_t* a, void* d_s, void* d_e, void* d_k1, void* d_ais, void* d_r1is,
                            void* d_r2is, void* d_ct0is) {
    HG_TRY({
        HG_CUDA(cudaSetDevice(ctx->dev.device));
        if (!qis || !k0is || !r1_bounds || !r2_bounds || !s || !e || !k1 || !a || !d_s || !d_e || !d_k1 || !d_ais || !d_r1is || !d_r2is || !d_ct0is)
            throw std::runtime_error("hg_bfv_witness_generate: NULL argument");
        with_field(ctx->field_id, [&](auto fp) {
            witness_generate<decltype(fp)>(ctx, n, K, qis, k0is, r1_bounds, r2_bounds, s, e, k1, a, d_s, d_e, d_k1, d_ais, d_r1is, d_r2is, d_ct0is);
        });
    })
}
int hg_mle_eval_host(int field_id, const uint64_t* table_limbs, size_t n, size_t num_vars, const uint64_t* point_ext, uint64_t* out_ext) {
    HG_TRY({
        if (n != (size_t)1 << num_vars) throw std::runtime_error("hg_mle_eval_host: the table must have 2^num_vars elements");
        with_field(field_id, [&](auto fp) {
            typedef decltype(fp) FP;
            std::vector<typename FP::B> t(n);
            for (size_t i = 0; i < n; i++) t[i] = FP::b_from_limbs(table_limbs + i * FP::B_LIMBS);
            std::vector<typename FP::X> pt(num_vars);
            for (size_t i = 0; i < num_vars; i++) pt[i] = FP::x_from_limbs(point_ext + i * FP::X_LIMBS);
            FP::x_to_limbs(GkrVerifierHost<FP>::mle_eval_base(t.data(), n, pt), out_ext);
        });
    })
}
void hg_circuit_free(hg_circuit* c) {
    if (!c) return;
    if (c->ctx) cudaSetDevice(c->ctx->dev.device);
    delete c;
}
int hg_circuit_insert_input(hg_circuit* c, size_t log2_size, size_t num_reps, int* out_id) {
    HG_TRY({ std::visit([&](auto& k) { *out_id = k.insert_input(log2_size, num_reps); }, c->c); })
}
int hg_circuit_insert_fft(hg_circuit* c, size_t log2_size, int inverse, int* out_id) {
    HG_TRY({ if (c->ctx) circuit_use_device(c); std::visit([&](auto& k) { *out_id = k.insert_fft(log2_size, inverse != 0); }, c->c); })
}
int hg_circuit_insert_lasso(hg_circuit* c, hg_lasso_node* node, int* out_id) {
    HG_TRY({
        if (!c->ctx) throw std::runtime_error("a host-only circuit takes its Lasso node through hg_circuit_insert_lasso_host");
        with_kind<GkrCircuitDev>(c, [&](auto& dc) { *out_id = dc.insert_lasso(&typed<field_t<decltype(dc)>>(node)); });
    })
}
int hg_circuit_insert_vanilla(hg_circuit* c, size_t input_arity, size_t log2_sub_input_size, size_t num_reps, size_t n_gates, const uint8_t* has_const,
                              const uint64_t* consts, const uint64_t* add_ptr, const uint64_t* add_coef, const uint32_t* add_input,
                              const uint64_t* add_wire, const uint64_t* mul_ptr, const uint64_t* mul_coef, const uint32_t* mul_in0, const uint64_t* mul_w0,
                              const uint32_t* mul_in1, const uint64_t* mul_w1, int* out_id) {
    HG_TRY({
        // every argument is checked before anything is read through it
        if (!c || !has_const || !consts || !add_ptr || !mul_ptr || !out_id || n_gates < 1) throw std::runtime_error("hg_circuit_insert_vanilla: NULL argument or no gates");
        // the edge arrays are sized by the CSR pointers: check those before anything is read through them
        if (add_ptr[0] != 0 || mul_ptr[0] != 0) throw std::runtime_error("hg_circuit_insert_vanilla: CSR pointers must start at 0");
        for (size_t g = 0; g < n_gates; g++)
            if (add_ptr[g + 1] < add_ptr[g] || mul_ptr[g + 1] < mul_ptr[g]) throw std::runtime_error("hg_circuit_insert_vanilla: CSR pointers must be non-decreasing");
        if (add_ptr[n_gates] > ((uint64_t)1 << 40) || mul_ptr[n_gates] > ((uint64_t)1 << 40)) throw std::runtime_error("hg_circuit_insert_vanilla: implausible edge count");
        if ((add_ptr[n_gates] && (!add_coef || !add_input || !add_wire)) || (mul_ptr[n_gates] && (!mul_coef || !mul_in0 || !mul_w0 || !mul_in1 || !mul_w1)))
            throw std::runtime_error("hg_circuit_insert_vanilla: NULL edge array");
        if (c->ctx) circuit_use_device(c);
        std::visit([&](auto& k) {
            const size_t L = field_t<decltype(k)>::B_LIMBS;  // limbs per coefficient
            VanillaDesc d;
            d.arity = input_arity; d.log2_sub = log2_sub_input_size; d.num_reps = num_reps; d.n_gates = n_gates;
            d.has_const.assign(has_const, has_const + n_gates);
            d.consts.assign(consts, consts + n_gates * L);
            d.add_ptr.assign(add_ptr, add_ptr + n_gates + 1);
            const size_t na = d.add_ptr[n_gates];
            d.add_coef.assign(add_coef, add_coef + na * L); d.add_in.assign(add_input, add_input + na); d.add_wire.assign(add_wire, add_wire + na);
            d.mul_ptr.assign(mul_ptr, mul_ptr + n_gates + 1);
            const size_t nm = d.mul_ptr[n_gates];
            d.mul_coef.assign(mul_coef, mul_coef + nm * L); d.mul_in0.assign(mul_in0, mul_in0 + nm); d.mul_w0.assign(mul_w0, mul_w0 + nm);
            d.mul_in1.assign(mul_in1, mul_in1 + nm); d.mul_w1.assign(mul_w1, mul_w1 + nm);
            *out_id = k.insert_vanilla(d);
        }, c->c);
    })
}
int hg_circuit_connect(hg_circuit* c, int from, int to) { HG_TRY({ std::visit([&](auto& k) { k.connect(from, to); }, c->c); }) }
int hg_circuit_evaluate(hg_circuit* c, const void* const* d_inputs, size_t n_inputs) {
    HG_TRY({
        circuit_use_device(c);
        with_kind<GkrCircuitDev>(c, [&](auto& dc) {
            typedef typename field_t<decltype(dc)>::B B;
            std::vector<const B*> v;
            for (size_t i = 0; i < n_inputs; i++) v.push_back((const B*)d_inputs[i]);
            dc.evaluate(v);
        });
    })
}
int hg_circuit_evaluate_host(hg_circuit* c, const void* const* host_inputs, const size_t* n_elems, size_t n_inputs) {
    HG_TRY({ circuit_use_device(c); with_kind<GkrCircuitDev>(c, [&](auto& dc) { evaluate_host(c, dc, host_inputs, n_elems, n_inputs); }); })
}
int hg_circuit_node_value(hg_circuit* c, int id, const void** d_ptr, size_t* len) {
    HG_TRY({
        circuit_use_device(c);
        with_kind<GkrCircuitDev>(c, [&](auto& dc) {
            if (id < 0 || (size_t)id >= dc.num_nodes()) throw std::runtime_error("no such node");
            *d_ptr = dc.node_value(id);
            *len = dc.node_out_len(id);
        });
    })
}
int hg_gkr_prove(hg_circuit* c, size_t n_output_claims, const size_t* point_lens, const uint64_t* points_ext, const uint64_t* values_ext,
                 hg_transcript* t, int mode) {
    HG_TRY({
        circuit_use_device(c);
        with_kind<GkrCircuitDev>(c, [&](auto& dc) {
            typedef field_t<decltype(dc)> FP;
            Keccak256Transcript<FP>& tr = typed<FP>(t);
            auto oc = claims_from_limbs<FP, typename GkrCircuitDev<FP>::InputClaim>(n_output_claims, point_lens, points_ext, values_ext);
            set_input_claims<FP>(c, dc.prove(tr, mode == HG_MODE_INTERACTIVE ? kModeInteractive : kModePrefetch, c->ctx->wire, oc));
        });
    })
}
void hg_gkr_timing(const hg_circuit* c, double* out_us6) {
    static const double host_only[6] = {0, 0, 0, 0, 0, 0};
    const double* t = c->ctx ? with_kind<GkrCircuitDev>(c, [](auto& dc) { return dc.timing(); }) : host_only;
    for (int i = 0; i < 6; i++) out_us6[i] = t[i];
}
size_t hg_gkr_num_challenges(const hg_circuit* c) { return c->ctx ? with_kind<GkrCircuitDev>(c, [](auto& dc) { return dc.total_challenges(); }) : 0; }
size_t hg_gkr_num_inputs(const hg_circuit* c) { return c->input_claims.size(); }
size_t hg_gkr_num_input_claims(const hg_circuit* c, size_t input) { return input < c->input_claims.size() ? c->input_claims[input].size() : 0; }
size_t hg_gkr_input_claim_num_vars(const hg_circuit* c, size_t input, size_t k) {  // 0 for an index out of range: no exception crosses the boundary
    if (!c || input >= c->input_claims.size() || k >= c->input_claims[input].size()) return 0;
    return c->input_claims[input][k].nvars;
}
int hg_gkr_input_claim(const hg_circuit* c, size_t input, size_t k, uint64_t* point_ext, uint64_t* value_ext) {
    HG_TRY({
        const auto& ic = c->input_claims.at(input).at(k);
        memcpy(point_ext, ic.point.data(), ic.point.size() * 8);
        memcpy(value_ext, ic.value.data(), ic.value.size() * 8);
    })
}

int hg_field_selftest(hg_ctx* ctx, int op, const uint64_t* a_ext, const uint64_t* b_ext, size_t n, uint64_t* out_ext) {
    HG_TRY({
        HG_CUDA(cudaSetDevice(ctx->dev.device));
        with_field(ctx->field_id, [&](auto fp) { field_selftest<decltype(fp)>(&ctx->dev, op, a_ext, b_ext, n, out_ext); });
    })
}

}  // extern "C"
