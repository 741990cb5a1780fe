// Device-resident Lasso node prover: orchestration of the kernels in kernels.cuh in the reference's protocol order
//   LassoNode::prove_claim_reduction            /root/reference/lasso/src/lasso.rs:57-114
//   prove_collation_sum_check                   /root/reference/lasso/src/lasso.rs:254-288
//   prove_memory_checking                       /root/reference/lasso/src/lasso.rs:292-339
//   MemoryCheckingProver::{new,prove}           /root/reference/lasso/src/memory_checking/prover.rs:35-89,158-181
//   prove_grand_product                         /root/reference/lasso/src/memory_checking/prover.rs:183-266
// The transcript stays on the host. Two modes (SURVEY.md 8b):
//   PREFETCH     all challenges are squeezed up front and uploaded once (legal because the reference transcript never
//                absorbs prover messages, transcript.rs:156,183-203); kernels run back to back, messages come back in
//                one copy at the end and are serialised in protocol order.
//   INTERACTIVE  one device->host->device round trip per squeeze; works with any transcript.
#pragma once
#include <cuda_runtime.h>
#include <nvtx3/nvToolsExt.h>

#include <array>
#include <chrono>
#include <functional>
#include <memory>
#include <string>
#include <vector>

#include "gkr_kernels.cuh"
#include "gp_fused.cuh"
#include "gp_kernels.cuh"
#include "kernels.cuh"
#include "lasso_host.hpp"
#include "transcript.hpp"

namespace hg {

struct CudaError : std::runtime_error { using std::runtime_error::runtime_error; };
// NVTX range named after the reference's tracing span (lasso.rs:57,156,253,291; sk_encryption_circuit.rs:442,455): Nsight / ncu --nvtx
// timelines of this library read like the reference's tracing-forest output. Header-only NVTX3: free when no tool is attached.
struct NvtxSpan {
    explicit NvtxSpan(const char* name) { nvtxRangePushA(name); }
    ~NvtxSpan() { nvtxRangePop(); }
    NvtxSpan(const NvtxSpan&) = delete;
    NvtxSpan& operator=(const NvtxSpan&) = delete;
};
#define HG_CUDA(expr)                                                                                            \
    do {                                                                                                         \
        cudaError_t _e = (expr);                                                                                 \
        if (_e != cudaSuccess) throw ::hg::CudaError(std::string(#expr) + ": " + cudaGetErrorString(_e));        \
    } while (0)
#define HG_LAUNCH_CHECK() HG_CUDA(cudaGetLastError())

// kernel classes for the per-class event timing bench.py reports (roofline of the dominant kernel)
enum KernelClass { KC_POLY = 0, KC_COUNTERS, KC_EQ, KC_DOT, KC_HASH, KC_TREE, KC_SC_COLL, KC_SC_GP, KC_MISC, KC_NTT, KC_GKR_PREP, KC_GKR_SC, KC_COUNT };
inline const char* kernel_class_name(int c) {
    static const char* n[] = {"polynomialize", "counters", "eq_build", "mle_dot", "hash_build", "product_tree", "sumcheck_collation",
                              "sumcheck_grand_product", "misc", "ntt", "gkr_layer_weights", "gkr_layer_sumcheck"};
    return (c >= 0 && c < KC_COUNT) ? n[c] : "?";
}
struct DeviceCtx {
    int device = 0;
    cudaStream_t stream = nullptr;    // the launching stream (KernelScope, HG_K and every helper read it at call time)
    cudaStream_t stream2 = nullptr;   // see hg_ctx_create
    cudaStream_t stream3 = nullptr;   // Lasso access counters next to the claim / collation sumcheck
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr, ev_fork3 = nullptr, ev_join3 = nullptr, ev_coll = nullptr;
    bool join3_pending = false;
    bool two_streams = true;
    int sm_count = 148;
    size_t launches = 0;  // kernels enqueued (bench.py "gpu_launches")
    // optional per-launch CUDA-event timing on the launching stream
    bool profile = false;
    struct Rec { int cls; cudaEvent_t a, b; size_t bytes; };
    std::vector<Rec> recs;
    size_t cls_launches[KC_COUNT] = {0};
    double cls_ms[KC_COUNT] = {0};
    size_t cls_bytes[KC_COUNT] = {0};
    void profile_reset() {
        for (auto& r : recs) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
        recs.clear();
        for (int i = 0; i < KC_COUNT; i++) { cls_launches[i] = 0; cls_ms[i] = 0; cls_bytes[i] = 0; }
    }
    void profile_collect() {
        cudaStreamSynchronize(stream);
        for (auto& r : recs) {
            float ms = 0;
            cudaEventElapsedTime(&ms, r.a, r.b);
            cls_launches[r.cls]++; cls_ms[r.cls] += ms; cls_bytes[r.cls] += r.bytes;
            cudaEventDestroy(r.a); cudaEventDestroy(r.b);
        }
        recs.clear();
    }
};
// brackets one kernel launch: counts it and, when profiling, times it with events on the launching stream
struct KernelScope {
    DeviceCtx* c; int cls; size_t bytes; cudaEvent_t a = nullptr, b = nullptr;
    KernelScope(DeviceCtx* ctx, int k, size_t algorithmic_bytes) : c(ctx), cls(k), bytes(algorithmic_bytes) {
        if (c->profile) { cudaEventCreate(&a); cudaEventCreate(&b); cudaEventRecord(a, c->stream); }
    }
    ~KernelScope() {
        c->launches++;
        if (c->profile) { cudaEventRecord(b, c->stream); c->recs.push_back({cls, a, b, bytes}); }
    }
};
#define HG_K(ctx, cls, bytes, ...)               \
    do {                                         \
        ::hg::KernelScope _ks(ctx, cls, bytes);  \
        __VA_ARGS__;                             \
        HG_LAUNCH_CHECK();                       \
    } while (0)

template <class T> struct DevBuf {
    T* p = nullptr;
    size_t n = 0;
    DevBuf() {}
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    ~DevBuf() { release(); }
    void alloc(size_t count) {
        release();
        if (count) HG_CUDA(cudaMalloc((void**)&p, count * sizeof(T)));
        n = count;  // only after the allocation succeeded: `buf.n < need` checks must not skip a retry
    }
    void release() { if (p) cudaFree(p); p = nullptr; n = 0; }
    size_t bytes() const { return n * sizeof(T); }
};
template <class T> struct PinnedBuf {
    T* p = nullptr;
    size_t n = 0;
    PinnedBuf() {}
    PinnedBuf(const PinnedBuf&) = delete;
    PinnedBuf& operator=(const PinnedBuf&) = delete;
    ~PinnedBuf() { if (p) cudaFreeHost(p); }
    void alloc(size_t count) {
        if (p) cudaFreeHost(p);
        p = nullptr; n = count;
        if (count) HG_CUDA(cudaMallocHost((void**)&p, count * sizeof(T)));
    }
};

// Upstream-format switches (SURVEY.md Appendix B). Host-only: the kernels always return values of the TRUE round
// polynomial; how they are put on the wire is decided here.
struct WireOptions {
    int a3_wire = 0;       // 0: coefficients c0,c2..cd   1: evaluations h(0),h(2)..h(d)
    int a3_h1 = 0;         // 0: h(1) := claim - h(0)     1: h(1) from the tables
    int a5_ascending = 1;  // distribute_powers: 1: sum_i b^i e_i   0: first expression gets the highest power
};
enum ProveMode { kModePrefetch = 0, kModeInteractive = 1 };

// ---------------------------------------------------------------------------------------------------------
// Challenge / message plumbing between the host transcript and the device pipeline.
template <class FP> class Channel {
  public:
    typedef typename FP::X X;
    struct RoundOp { void* st; size_t off, next_idx; WireOptions w; int slot_h1; bool round0; };  // arguments of one emit_round
    Channel(DeviceCtx* ctx, size_t chal_cap, size_t msg_cap) : ctx_(ctx) {
        d_chal_.alloc(chal_cap); h_chal_.alloc(chal_cap);
        d_msg_.alloc(msg_cap); h_msg_.alloc(msg_cap);
        HG_CUDA(cudaStreamCreateWithFlags(&copy_stream_, cudaStreamNonBlocking));
        HG_CUDA(cudaStreamCreateWithFlags(&copy_stream2_, cudaStreamNonBlocking));
        HG_CUDA(cudaEventCreateWithFlags(&ev_side_done_, cudaEventDisableTiming));
        HG_CUDA(cudaEventCreateWithFlags(&ev_side_copied_, cudaEventDisableTiming));
        HG_CUDA(cudaEventCreateWithFlags(&ev_early_copied_, cudaEventDisableTiming));
    }
    ~Channel() {
        cudaEventDestroy(ev_side_done_); cudaEventDestroy(ev_side_copied_); cudaEventDestroy(ev_early_copied_);
        cudaStreamDestroy(copy_stream_); cudaStreamDestroy(copy_stream2_);
    }
    Channel(const Channel&) = delete;
    Channel& operator=(const Channel&) = delete;
    void begin(Keccak256Transcript<FP>* tr, ProveMode mode, size_t total_chal) {
        tr_ = tr; active_tr_ = tr; mode_ = mode;
        chal_cursor_ = chal_ready_ = msg_cursor_ = msg_ready_ = 0;
        deferred_.clear(); deferred_done_ = 0;
        side_state_ = 0; early_armed_ = false;
        if (total_chal > d_chal_.n) throw std::runtime_error("Channel: challenge capacity exceeded");
        if (mode_ == kModePrefetch) {
            for (size_t i = 0; i < total_chal; i++) h_chal_.p[i] = tr_->squeeze_challenge();
            chal_ready_ = total_chal;
            HG_CUDA(cudaMemcpyAsync(d_chal_.p, h_chal_.p, total_chal * sizeof(X), cudaMemcpyHostToDevice, ctx_->stream));
        }
    }
    // index of the first of n consecutive challenges, squeezed at this point of the protocol
    size_t squeeze(size_t n = 1) {
        size_t first = chal_cursor_;
        chal_cursor_ += n;
        if (chal_cursor_ > d_chal_.n) throw std::runtime_error("Channel: challenge capacity exceeded");
        if (mode_ == kModeInteractive) {
            flush();
            for (size_t i = first; i < chal_cursor_; i++) h_chal_.p[i] = tr_->squeeze_challenge();
            chal_ready_ = chal_cursor_;
            HG_CUDA(cudaMemcpyAsync(d_chal_.p + first, h_chal_.p + first, n * sizeof(X), cudaMemcpyHostToDevice, ctx_->stream));
        } else if (chal_cursor_ > chal_ready_) {
            throw std::runtime_error("Channel: prefetch count too small");
        }
        return first;
    }
    size_t alloc_msg(size_t n) {
        size_t off = msg_cursor_;
        msg_cursor_ += n;
        if (msg_cursor_ > d_msg_.n) throw std::runtime_error("Channel: message capacity exceeded");
        return off;
    }
    void emit(std::function<void()> fn) { deferred_.emplace_back(); deferred_.back().fn = std::move(fn); }
    // a round message (emit_round): by far the most frequent serialiser (~1 500 per proof), kept as plain data instead of a
    // heap-allocated closure. `st` stays alive through the closures of its sumcheck that hold the shared_ptr.
    void emit_round_op(void (*exec)(Channel&, const RoundOp&), const RoundOp& op) { deferred_.emplace_back(); deferred_.back().exec = exec; deferred_.back().op = op; }
    // ---- side segment (prefetch mode): a run of messages whose serialisers depend on nothing emitted before them (the Lasso
    // node: it ignores its incoming claim, lasso.rs:60). Its messages are copied to the host as soon as its kernels finish and
    // serialised into a side buffer while the device works on what was enqueued after it; flush() splices the bytes in place.
    bool begin_side() {
        if (mode_ != kModePrefetch || side_state_ != 0 || tr_->hooked()) return false;  // a caller-owned transcript takes its messages one by one, in order
        side_state_ = 1; side_def_begin_ = deferred_.size(); side_msg_begin_ = msg_cursor_;
        return true;
    }
    void end_side() {  // call when every kernel of the segment has been enqueued
        if (side_state_ != 1) return;
        side_state_ = 2; side_def_end_ = deferred_.size(); side_msg_end_ = msg_cursor_;
        HG_CUDA(cudaEventRecord(ev_side_done_, ctx_->stream));
        HG_CUDA(cudaStreamWaitEvent(copy_stream_, ev_side_done_, 0));
        if (side_msg_end_ > side_msg_begin_)
            HG_CUDA(cudaMemcpyAsync(h_msg_.p + side_msg_begin_, d_msg_.p + side_msg_begin_, (side_msg_end_ - side_msg_begin_) * sizeof(X),
                                    cudaMemcpyDeviceToHost, copy_stream_));
        HG_CUDA(cudaEventRecord(ev_side_copied_, copy_stream_));
    }
    // ---- early head (prefetch mode, with a closed side segment): everything emitted BEFORE the side segment whose kernels are done
    // when `after` fires (the node sumchecks that precede the Lasso node in protocol order run on the second stream and finish long
    // before the grand products). Their messages are copied then, and flush() serialises them straight into the transcript while
    // the device still works on the side segment: about two thirds of the serialisation leaves the critical path.
    void arm_early(cudaEvent_t after) {
        if (side_state_ != 2 || side_msg_begin_ == 0 || side_def_begin_ == 0) return;
        HG_CUDA(cudaStreamWaitEvent(copy_stream2_, after, 0));
        HG_CUDA(cudaMemcpyAsync(h_msg_.p, d_msg_.p, side_msg_begin_ * sizeof(X), cudaMemcpyDeviceToHost, copy_stream2_));
        HG_CUDA(cudaEventRecord(ev_early_copied_, copy_stream2_));
        early_armed_ = true;
    }
    // bring finished messages to the host and serialise everything emitted so far, in order
    void flush(double* wait_us = nullptr, double* emit_us = nullptr) {
        auto now = []() { return std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
        const double t0 = now();
        double side_us = 0;
        if (side_state_ == 1) side_state_ = 0;  // never closed: plain in-order flush
        if (early_armed_ && side_state_ == 2 && deferred_done_ == 0 && msg_ready_ == 0) {
            HG_CUDA(cudaEventSynchronize(ev_early_copied_));
            const double e0 = now();
            msg_ready_ = side_msg_begin_;
            while (deferred_done_ < side_def_begin_) deferred_[deferred_done_++](*this);
            side_us += now() - e0;
        }
        early_armed_ = false;
        auto copy_range = [&](size_t a, size_t b) {
            if (b > a) HG_CUDA(cudaMemcpyAsync(h_msg_.p + a, d_msg_.p + a, (b - a) * sizeof(X), cudaMemcpyDeviceToHost, ctx_->stream));
        };
        if (side_state_ == 2) {
            copy_range(msg_ready_, side_msg_begin_);
            copy_range(side_msg_end_, msg_cursor_);
            HG_CUDA(cudaEventSynchronize(ev_side_copied_));
            const double s0 = now();
            Keccak256Transcript<FP> side;
            active_tr_ = &side;
            msg_ready_ = side_msg_end_;  // side serialisers read their own range only
            for (size_t i = side_def_begin_; i < side_def_end_; i++) deferred_[i](*this);
            active_tr_ = tr_;
            side_bytes_ = side.proof();
            side_state_ = 3;
            side_us += now() - s0;
        } else {
            copy_range(msg_ready_, msg_cursor_);
        }
        msg_ready_ = msg_cursor_;
        const double t1 = now();
        HG_CUDA(cudaStreamSynchronize(ctx_->stream));
        const double t2 = now();
        while (deferred_done_ < deferred_.size()) {
            if (side_state_ == 3 && deferred_done_ == side_def_begin_) {
                tr_->append_bytes(side_bytes_);
                deferred_done_ = side_def_end_;
                side_state_ = 0;
                continue;
            }
            deferred_[deferred_done_++](*this);
        }
        if (wait_us) *wait_us = (t1 - t0 - side_us) + (t2 - t1);
        if (emit_us) *emit_us = side_us + (now() - t2);
    }
    // ---- a proof split over several devices (LassoNodeDev::prove_shard): every device fills the message slots of the terms
    // it owns and leaves the others zero; the element-wise sum over devices is the message buffer of the whole proof
    void zero_messages() { HG_CUDA(cudaMemsetAsync(d_msg_.p, 0, d_msg_.bytes(), ctx_->stream)); }
    // copy this device's partial message buffer to `out`, host or device memory of the caller, WITHOUT serialising (the
    // serialisers stay queued for emit_merged). Stream-ordered, no host synchronisation. The caller sums the buffers of all
    // devices (hg_shard_merge, or k_shard_merge after an NCCL all-gather) and rank 0 hands the sum back to emit_merged
    size_t copy_partial_to(X* out, size_t cap) {
        if (msg_cursor_ > cap) throw std::runtime_error("Channel: shard message buffer too small");
        HG_CUDA(cudaMemcpyAsync(out, d_msg_.p, msg_cursor_ * sizeof(X), cudaMemcpyDefault, ctx_->stream));
        return msg_cursor_;
    }
    // replace the host copy of the messages by the merged one (host or device memory) and serialise
    void emit_merged(const X* merged, size_t count) {
        if (count != msg_cursor_) throw std::runtime_error("Channel: merged message count does not match this proof");
        HG_CUDA(cudaMemcpyAsync(h_msg_.p, merged, count * sizeof(X), cudaMemcpyDefault, ctx_->stream));
        HG_CUDA(cudaStreamSynchronize(ctx_->stream));
        msg_ready_ = msg_cursor_;
        for (; deferred_done_ < deferred_.size(); deferred_done_++) deferred_[deferred_done_](*this);
    }
    // ---- the serialisation of a sharded proof split over the devices too. The proof is the concatenation of what the serialisers
    // write, in order, and every device walked the whole protocol, so device `part` of `nparts` serialises one contiguous range of
    // serialisers into `out` and the ranges are concatenated by the caller. A range starts at the serialiser that initialises the
    // claim of a sumcheck (the round records behind it carry state from one to the next). Outside its range a device still runs the
    // plain serialisers (they move claim values between nodes) with their output discarded, and skips the round records, which are
    // ~95 % of the arithmetic: afterwards the input claims are valid on every device.
    void emit_merged_device_part(const X* d_merged, size_t count, int part, int nparts, std::vector<uint8_t>& out) {
        if (count != msg_cursor_) throw std::runtime_error("Channel: merged message count does not match this proof");
        if (nparts < 1 || part < 0 || part >= nparts) throw std::runtime_error("Channel: bad part index");
        if (tr_->hooked()) throw std::runtime_error("Channel: a sharded proof is serialised into the library's own transcript");
        HG_CUDA(cudaMemcpyAsync(h_msg_.p, d_merged, count * sizeof(X), cudaMemcpyDefault, ctx_->stream));
        // cut points: serialiser i may start a range if it is a plain one directly followed by a round record; weights = round records
        const size_t nd = deferred_.size();
        std::vector<size_t> cuts{0};
        std::vector<size_t> rounds_before(nd + 1, 0);
        for (size_t i = 0; i < nd; i++) rounds_before[i + 1] = rounds_before[i] + (deferred_[i].exec ? 1 : 0);
        for (size_t i = 1; i + 1 < nd; i++) if (!deferred_[i].exec && deferred_[i + 1].exec) cuts.push_back(i);
        cuts.push_back(nd);
        auto bound = [&](int q) -> size_t {  // first cut with at least q / nparts of the round records before it
            if (q <= 0) return 0;
            if (q >= nparts) return nd;
            const size_t want = rounds_before[nd] * (size_t)q / (size_t)nparts;
            for (size_t c : cuts) if (rounds_before[c] >= want) return c;
            return nd;
        };
        const size_t a = bound(part), b = bound(part + 1);
        HG_CUDA(cudaStreamSynchronize(ctx_->stream));
        msg_ready_ = msg_cursor_;
        Keccak256Transcript<FP> local, sink;
        sink.set_discard(true);
        for (size_t i = 0; i < nd; i++) {
            const bool mine = i >= a && i < b;
            active_tr_ = mine ? &local : &sink;
            dry_ = !mine;
            deferred_[i](*this);
        }
        dry_ = false;
        active_tr_ = tr_;
        deferred_done_ = nd;
        out = local.proof();
    }
    bool dry() const { return dry_; }
    size_t msg_used() const { return msg_cursor_; }
    const X* d_chal(size_t i) const { return d_chal_.p + i; }
    X* d_msg(size_t i) { return d_msg_.p + i; }
    X chal(size_t i) const { if (i >= chal_ready_) throw std::runtime_error("Channel: challenge not squeezed yet"); return h_chal_.p[i]; }
    X msg(size_t i) const { if (i >= msg_ready_) throw std::runtime_error("Channel: message not downloaded yet"); return h_msg_.p[i]; }
    Keccak256Transcript<FP>& transcript() { return *active_tr_; }
    bool prefetching() const { return mode_ == kModePrefetch; }
    size_t chal_used() const { return chal_cursor_; }
    size_t next_index() const { return chal_cursor_; }

  private:
    DeviceCtx* ctx_;
    Keccak256Transcript<FP>* tr_ = nullptr;
    Keccak256Transcript<FP>* active_tr_ = nullptr;  // where serialisers write: tr_, or the side buffer
    cudaStream_t copy_stream_ = nullptr, copy_stream2_ = nullptr;
    cudaEvent_t ev_side_done_ = nullptr, ev_side_copied_ = nullptr, ev_early_copied_ = nullptr;
    bool early_armed_ = false, dry_ = false;
    int side_state_ = 0;  // 0 none, 1 open, 2 closed (copy in flight), 3 serialised
    size_t side_def_begin_ = 0, side_def_end_ = 0, side_msg_begin_ = 0, side_msg_end_ = 0;
    std::vector<uint8_t> side_bytes_;
    ProveMode mode_ = kModePrefetch;
    DevBuf<X> d_chal_, d_msg_;
    PinnedBuf<X> h_chal_, h_msg_;
    size_t chal_cursor_ = 0, chal_ready_ = 0, msg_cursor_ = 0, msg_ready_ = 0;
    struct Deferred {
        std::function<void()> fn;
        void (*exec)(Channel&, const RoundOp&) = nullptr;
        RoundOp op;
        void operator()(Channel& ch) const { if (exec) { if (!ch.dry()) exec(ch, op); } else fn(); }
    };
    std::vector<Deferred> deferred_;
    size_t deferred_done_ = 0;
};

// ---------------------------------------------------------------------------------------------------------
// host arithmetic on round messages [UPSTREAM gkr::sum_check, assumptions A3]
template <class FP> struct RoundPoly {
    typedef typename FP::X X;
    static X small(u64 v) { return FP::lift(FP::b_from_u64(v)); }
    static X inv_small(int v) {  // 1/2, 1/3, 1/6 are needed every round: invert once
        static const X i2 = FP::x_inv(small(2)), i3 = FP::x_inv(small(3)), i6 = FP::x_mul(i2, i3);
        return v == 2 ? i2 : v == 3 ? i3 : i6;
    }
    // coefficients of the degree-d polynomial through (0,y0)..(d,yd), d in {1,2,3}, by forward differences
    static std::vector<X> interpolate(const std::vector<X>& y) {
        const int d = (int)y.size() - 1;
        if (d < 1 || d > 3) throw std::runtime_error("RoundPoly: unsupported degree");
        X d1 = FP::x_sub(y[1], y[0]);
        if (d == 1) return {y[0], d1};
        X d2 = FP::x_add(FP::x_sub(y[2], FP::x_add(y[1], y[1])), y[0]);
        X inv2 = inv_small(2);
        if (d == 2) {
            X c2 = FP::x_mul(d2, inv2);
            return {y[0], FP::x_sub(d1, c2), c2};
        }
        // d3 = y3 - 3y2 + 3y1 - y0
        X three = small(3);
        X d3 = FP::x_sub(FP::x_add(FP::x_sub(y[3], FP::x_mul(three, y[2])), FP::x_mul(three, y[1])), y[0]);
        X inv3 = inv_small(3), inv6 = inv_small(6);
        X c3 = FP::x_mul(d3, inv6);
        X h2 = FP::x_mul(d2, inv2), h3 = FP::x_mul(d3, inv2);
        X c2 = FP::x_sub(h2, h3);
        X c1 = FP::x_add(FP::x_sub(d1, h2), FP::x_mul(d3, inv3));
        return {y[0], c1, c2, c3};
    }
    static X horner(const std::vector<X>& c, X x) {
        X r = FP::x_zero();
        for (size_t i = c.size(); i-- > 0;) r = FP::x_add(FP::x_mul(r, x), c[i]);
        return r;
    }
};

// host-side state of one sumcheck instance (claim bookkeeping happens while messages are serialised)
template <class FP> struct ScHostState {
    typedef typename FP::X X;
    X claim;                         // the claim the WIRE polynomial is checked against (prove_sum_check's running claim)
    bool has_pending = false;
    X pending_wire[4];               // coefficients of the polynomial that went on the wire last round (degree pending_deg)
    X pending_true[4];               // coefficients of the TRUE round polynomial of the last round
    int pending_deg = 0;
    size_t pending_chal = 0;
    bool scaled = false;             // the device samples h / scale (phase 2 of a general layer: h = X(u) * the sampled polynomial)
    X scale;
};

struct ScScratch {
    void* partials = nullptr;  // X [max_blocks * max_batch * 4]
    unsigned* counters = nullptr;
    int max_blocks = 0;
    void* midpart = nullptr;   // X [HG_PROD_MID_K][midpart_segs][4]: CTA partial sums of the mid stage (k_prod_mid_one); nullptr: no mid stage
    size_t midpart_segs = 0;
};
// shared memory of k_prod_mid_one for nt input tables next to the weights
template <class FP> inline size_t prod_mid_smem(int nt) { return ((size_t)(nt + 1) * (HG_PROD_MID_SEG + HG_PROD_MID_SEG / 2) + (size_t)HG_PROD_MID_K * 8 * 3) * sizeof(typename FP::X); }

// serialisation of one round message + claim bookkeeping (runs on the host when the message has been downloaded).
// The device sends samples of the TRUE round polynomial h: h(0), h(inf), [h(-1)], and h(1) in round 0. With the running
// true sum s = h(0) + h(1) (= previous true polynomial at the previous challenge) they determine h; the wire message then
// follows the upstream format under assumptions A3 / A3'.
template <class FP, int D>
void emit_round(Channel<FP>& ch, std::shared_ptr<ScHostState<FP>> st, size_t off, const WireOptions& wo, bool round0, size_t next_idx,
                int slot_h1 = D) {
    typedef typename FP::X X;
    typename Channel<FP>::RoundOp rop;
    rop.st = st.get(); rop.off = off; rop.next_idx = next_idx; rop.w = wo; rop.slot_h1 = slot_h1; rop.round0 = round0;
    ch.emit_round_op([](Channel<FP>& chr, const typename Channel<FP>::RoundOp& o) {
        Channel<FP>* chp = &chr;
        ScHostState<FP>* st = (ScHostState<FP>*)o.st;
        const size_t off = o.off, next_idx = o.next_idx;
        const WireOptions w = o.w;
        const bool round0 = o.round0;
        const int slot_h1 = o.slot_h1;
        typedef RoundPoly<FP> RP;
        auto horner = [](const X* c, int deg, X x) { X r = c[deg]; for (int i = deg; i-- > 0;) r = FP::x_add(FP::x_mul(r, x), c[i]); return r; };
        auto sample = [&](size_t i) { const X v = chp->msg(i); return st->scaled ? FP::x_mul(v, st->scale) : v; };
        X s;
        if (round0) {
            s = FP::x_add(sample(off), sample(off + slot_h1));
        } else {
            X rprev = chp->chal(st->pending_chal);
            s = horner(st->pending_true, st->pending_deg, rprev);
            st->claim = horner(st->pending_wire, st->pending_deg, rprev);
        }
        const X h0 = sample(off), hinf = sample(off + 1);
        X tc[D + 1];
        tc[0] = h0;
        tc[D] = hinf;
        X a = FP::x_sub(FP::x_sub(s, FP::x_add(h0, h0)), hinf);  // sum of the middle coefficients
        if (D == 2) {
            tc[1] = a;
        } else {
            X bv = FP::x_add(FP::x_sub(sample(off + 2), h0), hinf);  // c2 - c1
            X inv2 = RP::inv_small(2);
            tc[2] = FP::x_mul(FP::x_add(a, bv), inv2);
            tc[1] = FP::x_mul(FP::x_sub(a, bv), inv2);
        }
        X co[D + 1];
        auto& tr = chp->transcript();
        if (w.a3_h1 == 0 && w.a3_wire == 0) {
            // default wire format: coefficients of the polynomial through (0, h(0)), (1, claim - h(0)), (k, h(k)) for k >= 2.
            // It differs from h by delta * L_1 with L_1 the Lagrange basis polynomial of node 1 over {0..D}:
            // D = 2: 2X - X^2;  D = 3: (6X - 5X^2 + X^3) / 2
            X h1 = tc[0];
            for (int k = 1; k <= D; k++) h1 = FP::x_add(h1, tc[k]);
            const X delta = FP::x_sub(FP::x_sub(st->claim, h0), h1);
            co[0] = tc[0];
            if (D == 2) {
                co[1] = FP::x_add(tc[1], FP::x_add(delta, delta));
                co[2] = FP::x_sub(tc[2], delta);
            } else {
                static const X k3 = RP::small(3), k52 = FP::x_mul(RP::small(5), RP::inv_small(2)), k12 = RP::inv_small(2);
                co[1] = FP::x_add(tc[1], FP::x_mul(delta, k3));
                co[2] = FP::x_sub(tc[2], FP::x_mul(delta, k52));
                co[3] = FP::x_add(tc[3], FP::x_mul(delta, k12));
            }
            tr.write_felt_ext(co[0]);
            for (int q = 2; q <= D; q++) tr.write_felt_ext(co[q]);
        } else {
            std::vector<X> tcv(tc, tc + D + 1), ev(D + 1);
            for (int k = 0; k <= D; k++) ev[k] = RP::horner(tcv, RP::small(k));
            std::vector<X> cov = tcv;
            if (w.a3_h1 == 0) {
                ev[1] = FP::x_sub(st->claim, ev[0]);
                cov = RP::interpolate(ev);
            }
            for (int k = 0; k <= D; k++) co[k] = cov[k];
            if (w.a3_wire == 0) { tr.write_felt_ext(co[0]); for (int q = 2; q <= D; q++) tr.write_felt_ext(co[q]); }
            else { tr.write_felt_ext(ev[0]); for (int q = 2; q <= D; q++) tr.write_felt_ext(ev[q]); }
        }
        for (int k = 0; k <= D; k++) { st->pending_wire[k] = co[k]; st->pending_true[k] = tc[k]; }
        st->pending_deg = D;
        st->pending_chal = next_idx;
        st->has_pending = true;
    }, rop);
}

// same for the fixed 4-slot layout [h(0), h(inf), h(-1), h(1)] of the generic GKR layer kernels (gkr_kernels.cuh)
template <class FP, int D>
void emit_round_slots(Channel<FP>& ch, std::shared_ptr<ScHostState<FP>> st, size_t off, const WireOptions& wo, bool round0, size_t next_idx) {
    emit_round<FP, D>(ch, st, off, wo, round0, next_idx, 3);
}

// one launch of k_sc_round with the right instantiation
template <class FP, int ARITY>
void launch_sc_round(DeviceCtx* ctx, int kclass, bool in_base, bool fold, const void* in, typename FP::X* out, size_t n_in, int nterm,
                     const typename FP::X* coeffs, const typename FP::X* r_prev, const ScScratch& sc, typename FP::X* msg) {
    typedef typename FP::B B;
    typedef typename FP::X X;
    size_t npairs = fold ? n_in / 4 : n_in / 2;
    int blocks = (int)std::min<size_t>((npairs + HG_BLOCK - 1) / HG_BLOCK, (size_t)sc.max_blocks);
    if (blocks < 1) blocks = 1;
    X* part = (X*)sc.partials;
    // algorithmic bytes of this launch: every input table read once, every folded table written once
    const size_t ntab = (size_t)nterm * ARITY;
    const size_t bytes = ntab * n_in * (in_base ? sizeof(B) : sizeof(X)) + (fold ? ntab * (n_in / 2) * sizeof(X) : 0);
    KernelScope _ks(ctx, kclass, bytes);
#define HG_SC(TIN, FOLD) \
    k_sc_round<FP, TIN, ARITY, FOLD><<<blocks, HG_BLOCK, 0, ctx->stream>>>((const TIN*)in, out, n_in, nterm, coeffs, r_prev, part, sc.counters, msg)
    if (in_base) { if (fold) HG_SC(B, true); else HG_SC(B, false); }
    else { if (!fold) throw std::runtime_error("launch_sc_round: extension input is always folded"); HG_SC(X, true); }
#undef HG_SC
    HG_LAUNCH_CHECK();
}

// prove_sum_check for g = t_0 * sum_i coeffs[i] * prod_{k<ARITY} t_{ARITY*i+k} over base tables of length n = 2^nv laid
// out back to back. Returns the message offset of the final evaluations and the index of the first round challenge.
template <class FP, int ARITY>
void sumcheck_dev(DeviceCtx* ctx, int kclass, Channel<FP>& ch, const WireOptions& wo, const typename FP::B* d_tables, size_t n, int nterm,
                  const typename FP::X* d_coeffs, typename FP::X* bufA, typename FP::X* bufB, const ScScratch& sc,
                  std::shared_ptr<ScHostState<FP>> st, size_t* first_chal, size_t* evals_off, bool launch = true, bool product_of_two = false) {
    typedef typename FP::B B;
    typedef typename FP::X X;
    constexpr int D = ARITY + 1;
    const int ntab = nterm * ARITY;
    int nv = 0;
    while (((size_t)1 << nv) < n) nv++;
    if (nv < 1) throw std::runtime_error("sumcheck_dev: num_vars must be positive");
    // g = t_0 * t_1 (the collation sumcheck: coefficients {0, 1}) with all challenges known: the last rounds run in one
    // shared-memory launch (k_prod_tail_one), the streamed rounds stop at jt
    const bool tail = product_of_two && ARITY == 1 && nterm == 2 && ch.prefetching() && nv >= 3;
    // with nv >= 12 the HG_PROD_MID_K rounds before the tail run in ONE launch on 1024-entry segments (k_prod_mid_one): streamed rounds
    // [0, js), mid rounds [js, jt), tail rounds [jt, nv)
    const bool mid = tail && nv >= 12 && sc.midpart != nullptr;
    const int js = !tail ? nv : (mid ? std::max(2, nv - 2 * HG_PROD_MID_K) : std::max(2, nv - HG_PROD_TAIL_LOG));
    const int jt = !tail ? nv : (mid ? js + HG_PROD_MID_K : js);
    const void* cur_in = d_tables;
    bool in_base = true;
    size_t n_in = n;
    size_t prev_chal = 0, tail_msg = 0, tail_chal = 0, mid_msg = 0, mid_chal = 0;
    for (int j = 0; j < nv; j++) {
        const bool streamed = j < js;
        size_t off = ch.alloc_msg(streamed ? (j == 0 ? D + 1 : D) : 4);  // the mid / tail kernels write 4 slots per round: [h(0), h(inf), -, 0]
        if (j == js) { mid_msg = off; mid_chal = prev_chal; }
        if (j == jt) { tail_msg = off; tail_chal = prev_chal; }
        if (streamed) {
            X* out = j == 0 ? nullptr : ((j & 1) ? bufA : bufB);
            if (launch && product_of_two && ARITY == 1 && nterm == 2) {  // g = t_0 * t_1: dedicated streaming kernel
                const size_t npairs = j == 0 ? n_in / 2 : n_in / 4;
                int blocks = (int)std::min<size_t>(std::max<size_t>(1, (npairs + HG_BLOCK * HG_COLL_PER_THREAD - 1) / (HG_BLOCK * HG_COLL_PER_THREAD)), (size_t)sc.max_blocks);
                KernelScope ks(ctx, kclass, 2 * n_in * (in_base ? sizeof(B) : sizeof(X)) + (j ? n_in * sizeof(X) : 0));
                if (j == 0) k_coll_round<FP, B, false><<<blocks, HG_BLOCK, 0, ctx->stream>>>(d_tables, nullptr, n_in, nullptr, (X*)sc.partials, sc.counters, ch.d_msg(off));
                else if (in_base) k_coll_round<FP, B, true><<<blocks, HG_BLOCK, 0, ctx->stream>>>((const B*)cur_in, out, n_in, ch.d_chal(prev_chal), (X*)sc.partials, sc.counters, ch.d_msg(off));
                else k_coll_round<FP, X, true><<<blocks, HG_BLOCK, 0, ctx->stream>>>((const X*)cur_in, out, n_in, ch.d_chal(prev_chal), (X*)sc.partials, sc.counters, ch.d_msg(off));
                HG_LAUNCH_CHECK();
            } else if (launch) {
                if (j == 0) launch_sc_round<FP, ARITY>(ctx, kclass, true, false, d_tables, nullptr, n, nterm, d_coeffs, nullptr, sc, ch.d_msg(off));
                else launch_sc_round<FP, ARITY>(ctx, kclass, in_base, true, cur_in, out, n_in, nterm, d_coeffs, ch.d_chal(prev_chal), sc, ch.d_msg(off));
            }
            if (j > 0) { cur_in = out; in_base = false; n_in >>= 1; }
        }
        const size_t next_idx = ch.next_index();  // the challenge squeezed right after this message
        emit_round<FP, D>(ch, st, off, wo, j == 0, next_idx);
        prev_chal = ch.squeeze(1);
        if (prev_chal != next_idx) throw std::runtime_error("sumcheck_dev: challenge index drift");
        if (j == 0 && first_chal) *first_chal = prev_chal;
    }
    // final evaluations: the tables now have 2 elements each
    size_t eo = ch.alloc_msg(ntab);
    if (evals_off) *evals_off = eo;
    if (!launch) return;
    if (tail) {
        ProdTailItem<FP> t;
        t.mid_part = nullptr; t.mid_msg = nullptr; t.mid_nseg = 0; t.mid_rounds = 0;
        if (mid) {
            ProdMidItem<FP> mi;
            mi.n_in = n_in; mi.nt = 1; mi.nseg = (int)(n_in / HG_PROD_MID_SEG);
            if (n_in < 2 * (size_t)HG_PROD_MID_SEG || (size_t)mi.nseg > sc.midpart_segs) throw std::runtime_error("sumcheck_dev: mid stage does not fit its scratch");
            X* obuf = (cur_in == (const void*)bufA) ? bufB : bufA;
            const size_t n_out = n_in >> HG_PROD_MID_K;
            mi.w_in = (const X*)cur_in; mi.tab_in = (const X*)cur_in + n_in; mi.w_out = obuf; mi.tab_out = obuf + n_out;
            mi.chal = ch.d_chal(mid_chal); mi.part = (X*)sc.midpart; mi.capture = nullptr; mi.cap_round = -1; mi.arity = 1;
            {
                KernelScope ks(ctx, kclass, 2 * n_in * sizeof(X));
                k_prod_mid_one<FP><<<mi.nseg, 256, prod_mid_smem<FP>(1), ctx->stream>>>(mi);
                HG_LAUNCH_CHECK();
            }
            t.mid_part = (const X*)sc.midpart; t.mid_msg = ch.d_msg(mid_msg); t.mid_nseg = mi.nseg; t.mid_rounds = HG_PROD_MID_K;
            cur_in = obuf;
            n_in = n_out;
        }
        t.w_in = (const X*)cur_in; t.tab_in = (const X*)cur_in + n_in; t.n_in = (int)n_in; t.nt = 1; t.rounds = nv - jt;
        t.chal = ch.d_chal(tail_chal); t.msg = ch.d_msg(tail_msg); t.evals = ch.d_msg(eo) + 1;  // evals[0] (= t_0) is not produced: the caller of the collation sumcheck discards both
        t.capture = nullptr; t.linear = 0; t.arity = 1; t.cap_round = -1;
        const size_t smem = ((size_t)2 * (n_in + n_in / 2) + 96) * sizeof(X);
        KernelScope ks(ctx, kclass, 2 * n_in * sizeof(X));
        k_prod_tail_one<FP><<<1, 256, smem, ctx->stream>>>(t);
        HG_LAUNCH_CHECK();
        return;
    }
    int blocks = (ntab + HG_BLOCK - 1) / HG_BLOCK;
    if (in_base) HG_K(ctx, kclass, 2 * ntab * sizeof(B), k_fold_final<FP, B><<<blocks, HG_BLOCK, 0, ctx->stream>>>((const B*)cur_in, ntab, ch.d_chal(prev_chal), ch.d_msg(eo)));
    else HG_K(ctx, kclass, 2 * ntab * sizeof(X), k_fold_final<FP, X><<<blocks, HG_BLOCK, 0, ctx->stream>>>((const X*)cur_in, ntab, ch.d_chal(prev_chal), ch.d_msg(eo)));
}

// one layer sumcheck recorded for batched execution (prefetch mode): everything the device needs is static
template <class FP> struct GpLayerJob {
    const typename FP::B* tables;  // [nvec][2n]
    size_t n;
    int nvec, nv;
    size_t gamma_idx, r0_idx, msg_off, evals_off;
    typename FP::X* coef = nullptr;          // [c_i | c_i * r_0], assigned by LassoNodeDev::prepare_gp_coeffs
    const typename FP::X* r0part = nullptr;  // round 0 sampled by the fused tree builders (gp_fused.cuh): [r0n][4] CTA partials
    int r0n = 0;
};

// Grand-product layer sumcheck with the specialised kernels of gp_kernels.cuh. tables: [nvec][2n] base elements.
// d_gamma: the layer's batching challenge (device); d_coeffs: scratch for [c_i | c_i * r_0] (2*nvec).
// *scaled = whether the final evaluations of l_i (i > 0) carry the factor c_i (true iff a round >= 1 ran).
template <class FP>
void gp_sumcheck_dev(DeviceCtx* ctx, Channel<FP>& ch, const WireOptions& wo, const typename FP::B* d_tables, size_t n, int nvec,
                     const typename FP::X* d_gamma, typename FP::X* d_coeffs, typename FP::X* bufA, typename FP::X* bufB, const ScScratch& sc,
                     std::shared_ptr<ScHostState<FP>> st, size_t* first_chal, size_t* evals_off, bool* scaled,
                     std::vector<GpLayerJob<FP>>* batch = nullptr, size_t gamma_idx = 0) {
    typedef typename FP::B B;
    typedef typename FP::X X;
    constexpr int D = 3;
    const int ntab = 2 * nvec;
    int nv = 0;
    while (((size_t)1 << nv) < n) nv++;
    if (batch) {
        // prefetch mode: only the protocol bookkeeping happens here; LassoNodeDev::run_gp_batch launches the work
        GpLayerJob<FP> job;
        job.tables = d_tables; job.n = n; job.nvec = nvec; job.nv = nv; job.gamma_idx = gamma_idx;
        for (int j = 0; j < nv; j++) {
            size_t off = ch.alloc_msg(j == 0 ? D + 1 : D);
            if (j == 0) job.msg_off = off;
            const size_t next_idx = ch.next_index();
            emit_round<FP, D>(ch, st, off, wo, j == 0, next_idx);
            size_t idx = ch.squeeze(1);
            if (j == 0) { job.r0_idx = idx; if (first_chal) *first_chal = idx; }
        }
        job.evals_off = ch.alloc_msg(ntab);
        if (evals_off) *evals_off = job.evals_off;
        if (scaled) *scaled = true;  // the batched kernels always pre-scale l_i (i > 0)
        batch->push_back(job);
        return;
    }
    X* part = (X*)sc.partials;
    X* d_c = d_coeffs;
    X* d_cr = d_coeffs + nvec;
    const int target_blocks = ctx->sm_count * 4;
    auto plan = [&](size_t threads_x, int* bx, int* groups, int* tpg) {
        size_t b = (threads_x + HG_BLOCK - 1) / HG_BLOCK;
        if (b < 1) b = 1;
        if (b > (size_t)sc.max_blocks) b = sc.max_blocks;
        int g = (int)std::min<size_t>((size_t)nvec, std::max<size_t>(1, ((size_t)target_blocks + b - 1) / b));
        *tpg = (nvec + g - 1) / g;
        *groups = (nvec + *tpg - 1) / *tpg;
        *bx = (int)b;
    };
    HG_K(ctx, KC_MISC, 0, k_gp_coeffs<FP><<<1, 32, 0, ctx->stream>>>(d_gamma, nullptr, nvec, wo.a5_ascending, d_c, d_cr));
    const void* cur_in = d_tables;
    bool in_base = true;
    size_t n_in = n, prev_chal = 0;
    for (int j = 0; j < nv; j++) {
        size_t off = ch.alloc_msg(j == 0 ? D + 1 : D);
        int bx, groups, tpg;
        if (j == 0) {
            constexpr int U = 4;
            plan((n / 2 + U - 1) / U, &bx, &groups, &tpg);
            KernelScope ks(ctx, KC_SC_GP, (size_t)ntab * n * sizeof(B));
            k_gp_r0<FP, U><<<dim3(bx, groups), HG_BLOCK, 0, ctx->stream>>>(d_tables, n, nvec, tpg, d_c, part, sc.counters, ch.d_msg(off));
            HG_LAUNCH_CHECK();
        } else {
            X* out = (j & 1) ? bufA : bufB;
            const X* rp = ch.d_chal(prev_chal);
            if (j == 1) HG_K(ctx, KC_MISC, 0, k_gp_coeffs<FP><<<1, 32, 0, ctx->stream>>>(d_gamma, rp, nvec, wo.a5_ascending, d_c, d_cr));
            plan(n_in / 4, &bx, &groups, &tpg);
            KernelScope ks(ctx, KC_SC_GP, (size_t)ntab * n_in * (in_base ? sizeof(B) : sizeof(X)) + (size_t)ntab * (n_in / 2) * sizeof(X));
            dim3 grid(bx, groups);
            if (in_base) k_gp_fold<FP, B, true><<<grid, HG_BLOCK, 0, ctx->stream>>>((const B*)cur_in, out, n_in, nvec, tpg, d_c, d_cr, rp, part, sc.counters, ch.d_msg(off));
            else k_gp_fold<FP, X, false><<<grid, HG_BLOCK, 0, ctx->stream>>>((const X*)cur_in, out, n_in, nvec, tpg, d_c, d_cr, rp, part, sc.counters, ch.d_msg(off));
            HG_LAUNCH_CHECK();
            cur_in = out; in_base = false; n_in >>= 1;
        }
        const size_t next_idx = ch.next_index();
        emit_round<FP, D>(ch, st, off, wo, j == 0, next_idx);
        prev_chal = ch.squeeze(1);
        if (prev_chal != next_idx) throw std::runtime_error("gp_sumcheck_dev: challenge index drift");
        if (j == 0 && first_chal) *first_chal = prev_chal;
    }
    size_t eo = ch.alloc_msg(ntab);
    int blocks = (ntab + HG_BLOCK - 1) / HG_BLOCK;
    if (in_base) HG_K(ctx, KC_SC_GP, 2 * ntab * sizeof(B), k_fold_final<FP, B><<<blocks, HG_BLOCK, 0, ctx->stream>>>((const B*)cur_in, ntab, ch.d_chal(prev_chal), ch.d_msg(eo)));
    else HG_K(ctx, KC_SC_GP, 2 * ntab * sizeof(X), k_fold_final<FP, X><<<blocks, HG_BLOCK, 0, ctx->stream>>>((const X*)cur_in, ntab, ch.d_chal(prev_chal), ch.d_msg(eo)));
    if (evals_off) *evals_off = eo;
    if (scaled) *scaled = !in_base;
}

template <class FP> __global__ void k_powers(const typename FP::X* __restrict__ base, int n, int ascending, typename FP::X* __restrict__ out) {
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    typename FP::X p = FP::x_one(), b = *base;
    for (int i = 0; i < n; i++) { out[ascending ? i : n - 1 - i] = p; p = FP::x_mul(p, b); }
}

// ---------------------------------------------------------------------------------------------------------
template <class FP> class LassoNodeDev {
  public:
    typedef typename FP::B B;
    typedef typename FP::X X;

    // LassoNode::new (lasso.rs:143-154). row_lookup[j] = index of row j's lookup type in preprocessing order.
    LassoNodeDev(DeviceCtx* ctx, const LassoPreprocessing& pp, int num_vars, const std::vector<uint8_t>& row_lookup)
        : ctx_(ctx), pp_(pp), num_vars_(num_vars), n_rows_(row_lookup.size()) {
        if (pp.lookups.size() > (size_t)HG_MAX_LOOKUPS - 1 || pp.num_memories > (size_t)HG_MAX_MEMORIES || pp.C > (size_t)HG_MAX_C)
            throw std::runtime_error("LassoNode: preprocessing exceeds device limits");
        log2M_ = (int)ilog2u(pp.M);
        if (log2M_ > 16 || log2M_ < 1) throw std::runtime_error("LassoNode: M must be in 2..=65536");
        R_ = (size_t)1 << num_vars;
        M_ = pp.M;
        if (n_rows_ > R_) throw std::runtime_error("LassoNode: more lookups than 2^num_vars");
        m_ = (int)pp.num_memories;
        // chunks: memories grouped by dimension, ascending (lasso.rs:303-336); chunk-major memory order (Q10)
        std::map<size_t, std::vector<size_t>> by_dim;
        for (size_t mi = 0; mi < pp.num_memories; mi++) by_dim[pp.memory_to_dimension_index[mi]].push_back(mi);
        std::vector<int> pos_mem, pos_dim, pos_slot, pos_sub;
        for (auto& kv : by_dim) {
            // F6: chunk `d` reads read_cts[d] / final_cts[d], i.e. the counters of MEMORY index d (lasso.rs:318-319)
            if (kv.first >= pp.num_memories) throw std::runtime_error("LassoNode: chunk index exceeds memory count (the reference panics here)");
            int slot = (int)chunk_dims_.size();
            chunk_dims_.push_back((int)kv.first);
            chunk_mems_.push_back(std::vector<int>(kv.second.begin(), kv.second.end()));
            for (size_t mi : kv.second) {
                pos_mem.push_back((int)mi); pos_dim.push_back((int)kv.first); pos_slot.push_back(slot);
                pos_sub.push_back((int)pp.memory_to_subtable_index[mi]);
            }
        }
        nslots_ = (int)chunk_dims_.size();
        pos_slot_host_ = pos_slot;

        NodeMeta meta;
        memset(&meta, 0, sizeof meta);
        meta.C = (int)pp.C; meta.log2M = log2M_; meta.num_lookups = (int)pp.lookups.size(); meta.num_memories = m_;
        for (size_t l = 0; l < pp.lookups.size(); l++) {
            unsigned tb = 0;
            for (unsigned b : pp.lookups[l]->chunk_bits(pp.M)) tb += b;
            meta.total_bits[l] = (u8)std::min(tb, 64u);
            auto& mem = pp.lookup_to_memory_indices[l];
            if (mem.size() > (size_t)HG_MAX_C) throw std::runtime_error("LassoNode: lookup uses too many memories");
            meta.lookup_nmem[l] = (u8)mem.size();
            for (size_t t = 0; t < mem.size(); t++) { meta.lookup_mem[l][t] = (u8)mem[t]; meta.mem_used[mem[t]] |= 1ULL << l; }
        }
        for (int mi = 0; mi < m_; mi++) { meta.mem_sub[mi] = (u8)pp.memory_to_subtable_index[mi]; meta.mem_dim[mi] = (u8)pp.memory_to_dimension_index[mi]; }
        for (int s = 0; s < nslots_; s++) slot_used_.push_back(meta.mem_used[chunk_dims_[s]]);
        for (int s = 0; s < nslots_; s++) slot_addr_dim_.push_back(meta.mem_dim[chunk_dims_[s]]);
        meta_host_ = meta;

        d_meta_.alloc(1);
        HG_CUDA(cudaMemcpy(d_meta_.p, &meta, sizeof meta, cudaMemcpyHostToDevice));
        d_row_lookup_.alloc(R_);
        {
            std::vector<uint8_t> rl(R_, 0xFF);
            std::copy(row_lookup.begin(), row_lookup.end(), rl.begin());
            for (auto v : row_lookup) if (v >= pp.lookups.size()) throw std::runtime_error("LassoNode: lookup index out of range");
            HG_CUDA(cudaMemcpy(d_row_lookup_.p, rl.data(), R_, cudaMemcpyHostToDevice));
        }
        // materialised subtables (lasso.rs:604-609), lifted with F::from(u64)
        {
            auto mats = pp.materialize_subtables();
            std::vector<B> flat(mats.size() * M_);
            for (size_t s = 0; s < mats.size(); s++) for (size_t i = 0; i < M_; i++) flat[s * M_ + i] = FP::b_from_u64(mats[s][i]);
            d_subtables_.alloc(flat.size());
            HG_CUDA(cudaMemcpy(d_subtables_.p, flat.data(), flat.size() * sizeof(B), cudaMemcpyHostToDevice));
        }
        auto up_int = [](DevBuf<int>& b, const std::vector<int>& v) { b.alloc(v.size()); HG_CUDA(cudaMemcpy(b.p, v.data(), v.size() * sizeof(int), cudaMemcpyHostToDevice)); };
        up_int(d_pos_mem_, pos_mem); up_int(d_pos_dim_, pos_dim); up_int(d_pos_slot_, pos_slot); up_int(d_pos_sub_, pos_sub);

        // work buffers
        d_dims_.alloc(pp.C * R_);
        d_E_.alloc((size_t)m_ * R_);
        d_coll_.alloc(2 * R_);  // [E_0 copy is not needed: table 0 of the collation is E_0 itself] -> coll = [E_0 | S]
        d_out_.alloc(R_);
        d_read_cts_.alloc((size_t)nslots_ * R_);
        d_final_cts_.alloc((size_t)nslots_ * M_);
        rows_per_block_ = 4096;
        nblk_cnt_ = (int)((std::max<size_t>(n_rows_, 1) + rows_per_block_ - 1) / rows_per_block_);
        if (nslots_ > HG_MAX_C) throw std::runtime_error("LassoNode: too many chunks");
        // counter scratch (radix sort of (address, row), kernels.cu): two element buffers, tile histograms, run boundaries
        cnt_cap_ = (size_t)nblk_cnt_ * rows_per_block_;
        d_cnt_a_.alloc((size_t)nslots_ * cnt_cap_);
        d_cnt_b_.alloc((size_t)nslots_ * cnt_cap_);
        d_cnt_hist_.alloc((size_t)2 * nslots_ * nblk_cnt_ * 256);  // tile histograms | their prefixes
        d_cnt_misc_.alloc((size_t)nslots_ * (512 + 8));           // digit starts, n_valid, digit totals
        d_cnt_runs_.alloc((size_t)2 * nslots_ * M_);              // start | end of every address run
        d_eq_.alloc(std::max(R_, M_));
        d_coeff_coll_.alloc(m_);
        d_wpow_.alloc((size_t)HG_MAX_LOOKUPS * HG_MAX_C);
        d_gp_coeffs_.alloc(4 * (size_t)m_ * (num_vars_ + log2M_ + 2) + 4);  // [c | c*r_0] per layer of both grand products
        // product trees: sum_k 2m * (N >> k) < 2m * 2N
        d_tree1_.alloc(2 * (size_t)m_ * 2 * R_);
        d_tree2_.alloc(2 * (size_t)m_ * 2 * M_);
        size_t nmax = std::max(R_, M_) / 2;  // longest sumcheck table
        d_bufA_.alloc(std::max<size_t>(4 * (size_t)m_ * (nmax / 2), 4 * (size_t)m_));
        d_bufB_.alloc(std::max<size_t>(4 * (size_t)m_ * (nmax / 4), 4 * (size_t)m_));
        // prefetch mode runs all layers concurrently: every layer needs its own fold buffers (L_2 and L_3 of its tables),
        // sum < 3/8 * 4m * (R + M) elements
        d_pool_.alloc(3 * (size_t)m_ * (R_ + M_) / 2 + 64);
        d_gp_partials_.alloc((size_t)ctx->sm_count * 64 * 4 + 4096);
        d_gp_counters_.alloc(64);  // one per layer of a batched round
        // CTA partial sums of the fused round 0 (gp_fused.cuh): <= sm_count*64 + 2m blocks per launch and layer, two layers per tree launch
        d_r0part_.alloc(4 * ((size_t)ctx->sm_count * 64 + 4 * (size_t)m_) * (size_t)(num_vars_ + log2M_ + 2));
        HG_CUDA(cudaMemset(d_gp_counters_.p, 0, d_gp_counters_.bytes()));
        h_desc_.alloc(1 << 16);
        d_desc_.alloc(1 << 16);
        {
            // grand-product tail kernel: tables of at most 2^GP_TAIL_LOG entries, every layer split over tail_groups_ CTAs by terms
            static_assert(FP::GP_TAIL_LOG >= 2 && FP::GP_TAIL_LOG <= HG_GP_TAIL_MAXR + 1, "GP_TAIL_LOG is out of the tail kernel's range");
            tail_groups_ = std::max(1, std::min((int)FP::GP_TAIL_GROUPS, 2 * m_));
            cudaFuncAttributes fa;  // the device's opt-in budget less the kernel's static shared memory (set_dynamic_smem_limits, abi.cu)
            HG_CUDA(cudaFuncGetAttributes(&fa, (const void*)k_gp_tail<FP>));
            const int smem_max = fa.maxDynamicSharedSizeBytes;
            while (gp_tail_smem(tail_groups_) > (size_t)smem_max && tail_groups_ < 2 * m_) tail_groups_++;  // more groups = fewer tables per CTA
            if (gp_tail_smem(tail_groups_) > (size_t)smem_max)
                throw std::runtime_error("LassoNode: the grand-product tail kernel needs " + std::to_string(gp_tail_smem(tail_groups_)) + " bytes of shared memory, the device offers " +
                                         std::to_string(smem_max));
            d_gp_tailpart_.alloc((size_t)(num_vars_ + log2M_ + 2) * tail_groups_ * (HG_GP_TAIL_MAXR + 1) * 4);
            d_gp_tailcnt_.alloc((size_t)(num_vars_ + log2M_ + 2));
            HG_CUDA(cudaMemset(d_gp_tailcnt_.p, 0, d_gp_tailcnt_.bytes()));
        }
        max_blocks_ = ctx->sm_count * 8;
        size_t batch = std::max<size_t>((size_t)m_, pp.C);
        d_partials_.alloc((size_t)max_blocks_ * 4 * batch);
        d_counters_.alloc(batch + 8);
        HG_CUDA(cudaMemset(d_counters_.p, 0, d_counters_.bytes()));
        sc_.partials = d_partials_.p; sc_.counters = d_counters_.p; sc_.max_blocks = max_blocks_;
        sc_.midpart_segs = std::max<size_t>(1, R_ / HG_PROD_MID_SEG);
        d_midpart_.alloc((size_t)HG_PROD_MID_K * sc_.midpart_segs * 4);
        sc_.midpart = d_midpart_.p;

        // challenge / message budget (SURVEY.md Appendix D)
        size_t v = num_vars_, lm = log2M_;
        total_chal_ = v + v + 2 + gp_chal_count(v) + gp_chal_count(lm);
        size_t msg = 1 + 4 * v + gp_msg_count(v) + gp_msg_count(lm) + pp.C + 2 * nslots_ + m_ + 16;
        msg_budget_ = msg;
        ch_.reset(new Channel<FP>(ctx, total_chal_ + 4, msg));

        // constant coefficient vectors
        {
            std::vector<B> cc(m_), wp((size_t)HG_MAX_LOOKUPS * HG_MAX_C, FP::b_zero());
            B w = FP::b_from_u64(pp.lookups.empty() ? M_ : pp.lookups[0]->combine_weight_base(pp.M));  // mock lookup = first in map order (lasso.rs:65)
            B p = FP::b_one();
            for (int i = 0; i < m_; i++) { cc[i] = p; p = FP::b_mul(p, w); }
            coll_coeff_host_ = cc;
            for (size_t l = 0; l < pp.lookups.size(); l++) {  // combine_lookups of lookup type l: operand t weighs w_l^t (range.rs:184-195: w = M)
                const B wl = FP::b_from_u64(pp.lookups[l]->combine_weight_base(pp.M));
                p = FP::b_one();
                for (int t = 0; t < HG_MAX_C; t++) { wp[l * HG_MAX_C + t] = p; p = FP::b_mul(p, wl); }
            }
            HG_CUDA(cudaMemcpy(d_wpow_.p, wp.data(), wp.size() * sizeof(B), cudaMemcpyHostToDevice));
        }
        // the uploads above are blocking cudaMemcpy calls from pageable memory (legacy stream); the proof kernels run on non-blocking
        // streams that do not wait for it, so make everything land now
        HG_CUDA(cudaDeviceSynchronize());
    }

    size_t device_bytes() const {
        return d_dims_.bytes() + d_E_.bytes() + d_coll_.bytes() + d_out_.bytes() + d_read_cts_.bytes() + d_final_cts_.bytes() + d_cnt_a_.bytes() + d_cnt_b_.bytes() +
               d_cnt_hist_.bytes() + d_cnt_runs_.bytes() + d_eq_.bytes() + d_tree1_.bytes() + d_tree2_.bytes() + d_bufA_.bytes() + d_bufB_.bytes() + d_pool_.bytes() + d_subtables_.bytes();
    }
    size_t num_rows() const { return n_rows_; }
    int num_vars() const { return num_vars_; }
    size_t total_challenges() const { return total_chal_; }

    // lasso.rs:57-114. d_inputs: device pointer, n_inputs base elements (the node's single input poly, lasso.rs:64).
    // Output: the claim (r, claimed_sum) for input 0 (lasso.rs:97,113).
    void prove(const B* d_inputs, size_t n_inputs, Keccak256Transcript<FP>& tr, ProveMode mode, const WireOptions& wo, std::vector<X>* out_point,
               X* out_value) {
        NvtxSpan span("LassoNode::prove_claim_reduction");
        if (!tr.prefetch_legal()) mode = kModeInteractive;  // a transcript that may absorb messages: one round trip per squeeze
        Channel<FP>& ch = *ch_;
        auto now = []() { return std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
        const double t_start = now();
        enqueue_witness(d_inputs, n_inputs, wo);
        ch.begin(&tr, mode, total_chal_);  // squeezing (Keccak on the host) overlaps the witness kernels, which need no challenges
        const double t_begin = now();
        size_t r_idx = 0, sum_off = 0;
        enqueue_protocol(ch, mode, wo, &r_idx, &sum_off);
        const double t_enq = now();
        ch.flush(&timing_[2], &timing_[3]);
        timing_[0] = t_begin - t_start;
        timing_[1] = t_enq - t_begin;
        if (ch.chal_used() != total_chal_) throw std::runtime_error("LassoNode: challenge count mismatch");
        if (out_point) { out_point->resize(num_vars_); for (int i = 0; i < num_vars_; i++) (*out_point)[i] = ch.chal(r_idx + i); }
        if (out_value) *out_value = ch.msg(sum_off);
    }

    // ---- one proof over `world` devices (SURVEY.md §8e). The round polynomials of the grand-product sumchecks are sums over
    // the 2m vectors (terms c_i * t_0 * l_i * r_i), the final evaluations / roots / openings belong to one vector or memory
    // each: device `rank` computes the terms it owns from its own copy of the witness, every message slot it does not own
    // stays zero, and the element-wise field sum of the message buffers over devices is the buffer a single device would
    // have produced. The challenges do not depend on the messages (SURVEY F3), so no device waits for another; the only
    // exchange is that one sum of `shard_message_count()` elements, after which rank 0 serialises (emit_shard).
    // Copies this device's partial message buffer to `out` (host or device memory of the caller, room for `cap` elements) on the
    // context's stream and returns its length; nothing waits for the device.
    size_t prove_shard(const B* d_inputs, size_t n_inputs, Keccak256Transcript<FP>& tr, const WireOptions& wo, int rank, int world, X* out, size_t cap) {
        if (world < 1 || rank < 0 || rank >= world || world > 2 * m_) throw std::runtime_error("LassoNode: bad shard rank / world size");
        if (!tr.prefetch_legal()) throw std::runtime_error("LassoNode: a sharded proof needs a transcript whose challenges do not depend on the messages");
        Channel<FP>& ch = *ch_;
        set_shard(rank, world);
        struct Reset { LassoNodeDev* n; ~Reset() { n->set_shard(0, 1); } } reset{this};
        enqueue_witness(d_inputs, n_inputs, wo);
        ch.zero_messages();
        ch.begin(&tr, kModePrefetch, total_chal_);
        enqueue_protocol(ch, kModePrefetch, wo, &shard_r_idx_, &shard_sum_off_);
        if (ch.chal_used() != total_chal_) throw std::runtime_error("LassoNode: challenge count mismatch");
        return ch.copy_partial_to(out, cap);
    }
    // rank 0, after prove_shard on the same node: write the proof from the merged message buffer (host or device memory)
    void emit_shard(const X* merged, size_t count, std::vector<X>* out_point, X* out_value) {
        Channel<FP>& ch = *ch_;
        ch.emit_merged(merged, count);
        if (out_point) { out_point->resize(num_vars_); for (int i = 0; i < num_vars_; i++) (*out_point)[i] = ch.chal(shard_r_idx_ + i); }
        if (out_value) *out_value = ch.msg(shard_sum_off_);
    }
    size_t shard_message_count() const { return msg_budget_; }
    // which device of a sharded proof this node works for (GkrCircuitDev::enqueue sets it around the node's two enqueue calls)
    void set_shard(int rank, int world) { shard_rank_ = rank; shard_world_ = world; }

    // polynomialize (lasso.rs:157-250): everything that needs no challenge
    void enqueue_witness(const B* d_inputs, size_t n_inputs, const WireOptions& wo) {
        NvtxSpan span("LassoNode::polynomialize");
        cudaStream_t s = ctx_->stream;
        const size_t R = R_, M = M_;
        const int m = m_;
        const size_t rows = std::min(n_inputs, n_rows_);  // izip! stops at the shorter (Q9)
        {
            size_t np2 = 1;  // lasso.rs:161 num_reads = inputs.len().next_power_of_two(); lasso.rs:79-80 assert_eq!(num_vars, self.num_vars)
            while (np2 < n_inputs) np2 <<= 1;
            if (np2 != R_) throw std::runtime_error("assertion `left == right` failed: num_vars of the input does not match the node (lasso.rs:80)");
        }

        // collation coefficients (A5): uploaded when the option changes, not per proof
        if (coll_coeff_state_ != (wo.a5_ascending ? 1 : 2)) {
            std::vector<B> cc = coll_coeff_host_;
            if (!wo.a5_ascending) std::reverse(cc.begin(), cc.end());
            HG_CUDA(cudaMemcpyAsync(d_coeff_coll_.p, cc.data(), cc.size() * sizeof(B), cudaMemcpyHostToDevice, s));
            X one_one[2] = {FP::x_zero(), FP::x_one()};  // g(E_0, S) = E_0 * (0 * E_0 + 1 * S), see enqueue_protocol
            if (!d_coll_terms_.n) d_coll_terms_.alloc(2);
            HG_CUDA(cudaMemcpyAsync(d_coll_terms_.p, one_one, sizeof one_one, cudaMemcpyHostToDevice, s));
            HG_CUDA(cudaStreamSynchronize(s));  // stack temporaries
            coll_coeff_state_ = wo.a5_ascending ? 1 : 2;
        }
        // ---- polynomialize (lasso.rs:157-250)
        B* d_S = d_coll_.p + R;
        HG_K(ctx_, KC_POLY, R * (sizeof(B) + 1 + pp_.C * 2 + ((size_t)m + 2) * sizeof(B)),
             k_polynomialize<FP><<<(unsigned)((R + HG_BLOCK - 1) / HG_BLOCK), HG_BLOCK, 0, s>>>(d_inputs, rows, d_row_lookup_.p, d_meta_.p, d_subtables_.p,
                                                                                                d_coeff_coll_.p, d_wpow_.p, R, d_dims_.p, d_E_.p, d_S, d_out_.p));
        HG_CUDA(cudaMemcpyAsync(d_coll_.p, d_E_.p, R * sizeof(B), cudaMemcpyDeviceToDevice, s));
        // access counters: needed only by the hash build (after gamma, tau), so they run on a side stream next to the claim
        // evaluation and the collation sumcheck; enqueue_protocol joins before the first kernel that reads them
        const bool side = ctx_->two_streams && !ctx_->profile && ctx_->stream3 != nullptr;
        cudaStream_t cs = s;
        struct StreamRestore {  // an exception between here and the join must not leave the context launching on stream3
            DeviceCtx* c; cudaStream_t main;
            ~StreamRestore() { c->stream = main; }
        } restore{ctx_, s};
        if (side) {
            HG_CUDA(cudaEventRecord(ctx_->ev_fork3, s));
            HG_CUDA(cudaStreamWaitEvent(ctx_->stream3, ctx_->ev_fork3, 0));
            cs = ctx_->stream3;
            ctx_->stream = cs;  // HG_K times / counts on the launching stream
        }
        HG_CUDA(cudaMemsetAsync(d_read_cts_.p, 0, d_read_cts_.bytes(), cs));
        {
            CntSlots sl;
            for (int q = 0; q < HG_MAX_C; q++) { sl.addr[q] = nullptr; sl.used[q] = 0; }
            for (int q = 0; q < nslots_; q++) { sl.addr[q] = d_dims_.p + (size_t)slot_addr_dim_[q] * R; sl.used[q] = slot_used_[q]; }
            // stable radix sort of (address, row) by the low then the high address byte; counters from the run boundaries
            u32* d_digit_start = d_cnt_misc_.p;
            u32* d_nvalid = d_cnt_misc_.p + (size_t)nslots_ * 256;
            u32* d_cnt_base = d_cnt_hist_.p + (size_t)nslots_ * nblk_cnt_ * 256;
            u32* d_digit_total = d_cnt_misc_.p + (size_t)nslots_ * 256 + 8;
            u32* d_start = d_cnt_runs_.p;
            u32* d_end = d_cnt_runs_.p + (size_t)nslots_ * M;
            HG_CUDA(cudaMemsetAsync(d_cnt_runs_.p, 0, d_cnt_runs_.bytes(), cs));
            // a device of a sharded proof counts only the chunk slots its vectors (and its share of the openings) read
            SlotMap sm;
            int ns = 0;
            for (int q = 0; q < HG_MAX_C; q++) sm.s[q] = 0;
            for (int q = 0; q < nslots_; q++) if (slot_needed(q)) sm.s[ns++] = q;
            const dim3 tiles(nblk_cnt_, ns);
            // algorithmic bytes of the class (booked on the first launch): address column and lookup type read once, both
            // counter tables written once. The sort scratch (~3x that) is traffic, not algorithm (DESIGN.md section 5).
            const size_t cnt_alg = (size_t)ns * (rows * (2 + 1 + 4) + M * 4);
            for (int pass = 0; pass < 2 && ns > 0; pass++) {
                const u64* src = pass == 0 ? nullptr : d_cnt_a_.p;
                u64* dst = pass == 0 ? d_cnt_a_.p : d_cnt_b_.p;
                HG_K(ctx_, KC_COUNTERS, pass == 0 ? cnt_alg : 0,
                     k_cnt_digit_hist<<<tiles, 1024, 0, cs>>>(sm, pass, sl, d_row_lookup_.p, rows, cnt_cap_, src, d_nvalid, nblk_cnt_, d_cnt_hist_.p));
                HG_K(ctx_, KC_COUNTERS, 0, k_cnt_digit_scan<<<dim3(8, ns), 1024, 0, cs>>>(sm, nblk_cnt_, d_cnt_hist_.p, d_cnt_base, d_digit_total));
                HG_K(ctx_, KC_COUNTERS, 0, k_cnt_digit_starts<<<ns, 256, 0, cs>>>(sm, d_digit_total, d_digit_start, d_nvalid));
                HG_K(ctx_, KC_COUNTERS, 0,
                     k_cnt_digit_scatter<<<tiles, 1024, 0, cs>>>(sm, pass, sl, d_row_lookup_.p, rows, cnt_cap_, src, d_nvalid, nblk_cnt_, d_cnt_base, d_digit_start, dst));
            }
            const unsigned fin_blocks = (unsigned)((std::max<size_t>(cnt_cap_, M) + 255) / 256);
            if (ns > 0) {
                HG_K(ctx_, KC_COUNTERS, 0, k_cnt_heads<<<dim3(fin_blocks, ns), 256, 0, cs>>>(sm, cnt_cap_, d_cnt_b_.p, d_nvalid, M, d_start, d_end));
                HG_K(ctx_, KC_COUNTERS, 0,
                     k_cnt_finish<<<dim3(fin_blocks, ns), 256, 0, cs>>>(sm, cnt_cap_, d_cnt_b_.p, d_nvalid, M, d_start, d_end, R, d_read_cts_.p, d_final_cts_.p));
            }
        }
        if (side) {
            ctx_->stream = s;
            HG_CUDA(cudaEventRecord(ctx_->ev_join3, cs));
            ctx_->join3_pending = true;
        }
    }

    // the interactive part of prove_claim_reduction on an already-begun channel (lasso.rs:85-113)
    void enqueue_protocol(Channel<FP>& ch, ProveMode mode, const WireOptions& wo, size_t* out_r_idx, size_t* out_sum_off) {
        cudaStream_t s = ctx_->stream;
        const size_t R = R_, M = M_;
        const int m = m_, v = num_vars_;
        // ---- r, claimed sum (lasso.rs:85, :264, :269)
        const size_t r_idx = ch.squeeze(v);
        const size_t sum_off = ch.alloc_msg(1);
        const bool lead = shard_rank_ == 0;  // the claim and the collation sumcheck belong to rank 0 (the openings are distributed, see below)
        // With every challenge known up front nothing below waits for the claim or the collation sumcheck (gamma, tau are challenges), so
        // they run on the side stream behind the access counters, next to the hash / tree / grand-product kernels, and are joined before
        // the openings (which reuse the eq tables and the partial-sum scratch). Measured: no change of the single-proof latency (5.07 vs
        // 5.08 ms, profiles/r2_experiments.md) because the three streams already keep the SMs busy, so a single-device proof keeps them
        // on the main stream. A sharded proof is latency-bound on every rank and rank 0 alone runs these two: there the side stream is used.
        const bool coll_side = shard_world_ > 1 && lead && mode == kModePrefetch && ctx_->two_streams && !ctx_->profile && ctx_->stream3 != nullptr && ctx_->ev_coll != nullptr;
        struct CollStream {  // launches go to stream3 while this lives (RAII: an exception must not leave the context there)
            DeviceCtx* c; cudaStream_t main; bool on;
            CollStream(DeviceCtx* ctx, bool enable) : c(ctx), main(ctx->stream), on(enable) {
                if (!on) return;
                cudaEventRecord(c->ev_fork3, main);  // everything enqueued so far (challenge upload, polynomialize) precedes the side work
                cudaStreamWaitEvent(c->stream3, c->ev_fork3, 0);
                c->stream = c->stream3;
            }
            void end() { if (on) { cudaEventRecord(c->ev_coll, c->stream3); c->stream = main; on = false; } }
            ~CollStream() { if (on) c->stream = main; }
        } coll_stream(ctx_, coll_side);
        if (lead) eval_tables<B>(ch, d_out_.p, R, 1, R, r_idx, v, sum_off);
        auto coll_state = std::make_shared<ScHostState<FP>>();
        {
            Channel<FP>* chp = &ch;
            ch.emit([chp, coll_state, sum_off]() {
                X cs = chp->msg(sum_off);
                chp->transcript().write_felt_ext(cs);
                coll_state->claim = cs;
            });
        }
        // ---- collation sumcheck (lasso.rs:271-279): t_0 * sum_i c_i t_i == E_0 * S with S = sum_i c_i E_i
        {
            NvtxSpan span("LassoNode::prove_collation_sum_check");
            // g(E_0, S) = E_0 * (0 * E_0 + 1 * S): nterm = 2, arity 1, tables [E_0 | S]; coefficients {0, 1} live in d_coll_terms_
            sumcheck_dev<FP, 1>(ctx_, KC_SC_COLL, ch, wo, d_coll_.p, R, 2, d_coll_terms_.p, d_bufA_.p, d_bufB_.p, sc_, coll_state, nullptr, nullptr, lead, true);
        }
        coll_stream.end();
        // ---- gamma, tau (lasso.rs:99)
        NvtxSpan span_mc("LassoNode::prove_memory_checking");
        const size_t gt_idx = ch.squeeze(2);
        if (ctx_->join3_pending) {  // the access counters (enqueue_witness) are read from here on
            HG_CUDA(cudaStreamWaitEvent(s, ctx_->ev_join3, 0));
            ctx_->join3_pending = false;
        }
        // ---- memory checking (lasso.rs:292-339, prover.rs:35-181)
        const bool fused_up = R >= 4;  // hash build fused with the first tree level
        size_t x_idx = 0, y_idx = 0;
        std::vector<GpLayerJob<FP>> jobs;
        GpPlan plan1, plan2;
        bool fuse_hash = false;
        if (mode == kModePrefetch) {
            // all challenges are on the device already: do the protocol bookkeeping of both grand products first (message
            // slots, challenge indices), then launch coefficients -> hashes -> trees (+ round 0) -> rounds >= 1
            grand_product(ch, wo, d_tree1_.p, R, &x_idx, &jobs, fused_up, &plan1);
            grand_product(ch, wo, d_tree2_.p, M, &y_idx, &jobs, false, &plan2);
            prepare_gp_coeffs(ch, wo, jobs);
            fuse_hash = fused_up && gp_needs_r0(R, 0, plan1.nvars);
        }
        if (fuse_hash) {
            GpLayerJob<FP>& j0 = jobs[plan1.job_begin + plan1.nvars - 2];  // the sumcheck on layer 0
            const size_t work = R / 4;                                      // row pairs per memory
            const int nxb = fused_nxb(work, m);
            X* part = r0_alloc((size_t)nxb * m);
            j0.r0part = part; j0.r0n = nxb * m;
            HG_K(ctx_, KC_HASH, 0, k_hash_t0<FP><<<(unsigned)((R / 4 + HG_BLOCK - 1) / HG_BLOCK), HG_BLOCK, 0, s>>>(d_dims_.p, d_read_cts_.p, d_E_.p, d_pos_mem_.p, d_pos_dim_.p,
                                                                                                                d_pos_slot_.p, ch.d_chal(gt_idx), R, d_tree1_.p));
            HG_K(ctx_, KC_HASH, (size_t)m * R * (2 + 4 + 4 * sizeof(B)),
                 k_hash_rw_up_r0<FP><<<nxb * m, HG_FUSED_BLOCK, 0, s>>>(d_dims_.p, d_read_cts_.p, d_E_.p, d_pos_mem_.p, d_pos_dim_.p, d_pos_slot_.p, ch.d_chal(gt_idx), R, m,
                                                                      d_tree1_.p, d_tree1_.p + (size_t)2 * m * R, own_range(2 * m), j0.coef, part, nxb));
        } else if (fused_up) {
            HG_K(ctx_, KC_HASH, (size_t)m * R * (2 + 4 + 4 * sizeof(B)),
                 k_hash_rw_up<FP><<<dim3((unsigned)((R / 4 + HG_BLOCK - 1) / HG_BLOCK + (R < 4 ? 1 : 0)), m), HG_BLOCK, 0, s>>>(
                     d_dims_.p, d_read_cts_.p, d_E_.p, d_pos_mem_.p, d_pos_dim_.p, d_pos_slot_.p, ch.d_chal(gt_idx), R, m, d_tree1_.p,
                     d_tree1_.p + (size_t)2 * m * R, own_range(2 * m)));
        } else {
            HG_K(ctx_, KC_HASH, (size_t)m * R * (2 + 4 + 3 * sizeof(B)),
                 k_hash_rw<FP><<<dim3((unsigned)((R + HG_BLOCK - 1) / HG_BLOCK), m), HG_BLOCK, 0, s>>>(d_dims_.p, d_read_cts_.p, d_E_.p, d_pos_mem_.p, d_pos_dim_.p,
                                                                                                       d_pos_slot_.p, ch.d_chal(gt_idx), R, m, d_tree1_.p));
        }
        HG_K(ctx_, KC_HASH, (size_t)m * M * (4 + 3 * sizeof(B)),
             k_hash_if<FP><<<dim3((unsigned)((M + HG_BLOCK - 1) / HG_BLOCK), m), HG_BLOCK, 0, s>>>(d_subtables_.p, d_final_cts_.p, d_pos_sub_.p, d_pos_slot_.p,
                                                                                                   ch.d_chal(gt_idx), M, m, d_tree2_.p, own_range(2 * m)));
        if (mode == kModePrefetch) {
            build_trees(ch, plan1, plan2, jobs);
            run_gp_batch(ch, wo, jobs);
        } else {
            grand_product(ch, wo, d_tree1_.p, R, &x_idx, nullptr, fused_up);
            grand_product(ch, wo, d_tree2_.p, M, &y_idx, nullptr, false);
        }
        // ---- openings (prover.rs:173-178, mod.rs:80-93)
        const size_t o_dims = ch.alloc_msg(pp_.C), o_rts = ch.alloc_msg(nslots_), o_fcs = ch.alloc_msg(nslots_), o_e = ch.alloc_msg(m);
        if (coll_side) HG_CUDA(cudaStreamWaitEvent(s, ctx_->ev_coll, 0));  // claim + collation sumcheck done: their scratch is free, their messages are in
        build_eq(ch, x_idx, v);
        {   // dim(x) openings and E_i(x) openings: tables split evenly over the devices
            const int c0 = (int)(pp_.C * shard_rank_ / shard_world_), c1 = (int)(pp_.C * (shard_rank_ + 1) / shard_world_);
            if (c1 > c0) dot_tables<u16>(ch, d_dims_.p + (size_t)c0 * R, R, c1 - c0, R, o_dims + c0);
            const int e0 = (int)((size_t)m * shard_rank_ / shard_world_), e1 = (int)((size_t)m * (shard_rank_ + 1) / shard_world_);
            if (e1 > e0) dot_tables<B>(ch, d_E_.p + (size_t)e0 * R, R, e1 - e0, R, o_e + e0);
        }
        // read_ts(x) / final_cts(y) of a chunk slot: on the device that owns the slot's first read vector (it has the counters)
        if (shard_world_ == 1) {
            dot_tables<u32>(ch, d_read_cts_.p, R, nslots_, R, o_rts);
            build_eq(ch, y_idx, log2M_);
            dot_tables<u32>(ch, d_final_cts_.p, M, nslots_, M, o_fcs);
        } else {
            bool any = false;
            for (int q = 0; q < nslots_; q++) if (slot_owner(q) == shard_rank_) { dot_tables<u32>(ch, d_read_cts_.p + (size_t)q * R, R, 1, R, o_rts + q); any = true; }
            if (any) {
                build_eq(ch, y_idx, log2M_);
                for (int q = 0; q < nslots_; q++) if (slot_owner(q) == shard_rank_) dot_tables<u32>(ch, d_final_cts_.p + (size_t)q * M, M, 1, M, o_fcs + q);
            }
        }
        {
            Channel<FP>* chp = &ch;
            auto dims = chunk_dims_; auto mems = chunk_mems_;
            ch.emit([chp, dims, mems, o_dims, o_rts, o_fcs, o_e]() {
                auto& t = chp->transcript();
                for (size_t c = 0; c < dims.size(); c++) {
                    t.write_felt_ext(chp->msg(o_dims + dims[c]));
                    t.write_felt_ext(chp->msg(o_rts + c));
                    t.write_felt_ext(chp->msg(o_fcs + c));
                    for (int mi : mems[c]) t.write_felt_ext(chp->msg(o_e + mi));
                }
            });
        }
        *out_r_idx = r_idx;
        *out_sum_off = sum_off;
    }
    size_t message_budget() const { return msg_budget_; }

    // test hooks: copies of the polynomialised witness
    void download_polys(std::vector<u16>* dims, std::vector<u32>* read_cts, std::vector<u32>* final_cts, std::vector<B>* E) {
        HG_CUDA(cudaStreamSynchronize(ctx_->stream));
        auto dl = [](auto* vec, auto& buf) { vec->resize(buf.n); HG_CUDA(cudaMemcpy(vec->data(), buf.p, buf.bytes(), cudaMemcpyDeviceToHost)); };
        if (dims) dl(dims, d_dims_);
        if (read_cts) dl(read_cts, d_read_cts_);
        if (final_cts) dl(final_cts, d_final_cts_);
        if (E) dl(E, d_E_);
    }
    const std::vector<int>& chunk_dims() const { return chunk_dims_; }
    // host-side phases of the last prove in microseconds: squeeze+upload challenges, enqueue kernels, wait for the GPU, serialise
    const double* timing() const { return timing_; }

  private:
    static size_t gp_chal_count(size_t nvars) {  // layers nv = 0..nvars-1: mu each; gamma + nv round challenges for nv >= 1
        size_t c = 0;
        for (size_t nv = 0; nv < nvars; nv++) c += 1 + (nv ? 1 + nv : 0);
        return c;
    }
    size_t gp_msg_count(size_t nvars) const {
        size_t c = 2 * (size_t)m_;  // roots
        for (size_t nv = 0; nv < nvars; nv++) c += 4 * (size_t)m_ + 4 * nv;
        return c;
    }
    static int eq_lo_bits(int nv) { return nv < 12 ? nv : 12; }
    void build_eq(Channel<FP>& ch, size_t point_idx, int nv) {
        const int lo = eq_lo_bits(nv);
        eq_nv_ = nv;
        size_t n = ((size_t)1 << lo) + ((size_t)1 << (nv - lo));
        HG_K(ctx_, KC_EQ, n * sizeof(X), k_eq_split<FP><<<(unsigned)((n + HG_BLOCK - 1) / HG_BLOCK), HG_BLOCK, 0, ctx_->stream>>>(ch.d_chal(point_idx), nv, lo, d_eq_.p, d_eq_.p + ((size_t)1 << lo)));
    }
    template <class T> void dot_tables(Channel<FP>& ch, const T* tables, size_t stride, int ntab, size_t n, size_t msg_off) {
        const int lo = eq_lo_bits(eq_nv_);
        if (n != (size_t)1 << eq_nv_) throw std::runtime_error("dot_tables: eq tables were built for another size");
        // about 6 CTAs per SM over all tables of the launch: every CTA ends with a block-level reduction that costs as much as
        // ~100 elements per thread, so few long CTAs beat many short ones
        const size_t per_table = std::max<size_t>(1, ((size_t)ctx_->sm_count * 6 + ntab - 1) / ntab);
        int blocks = (int)std::min<size_t>(n >> lo, std::min<size_t>(per_table, (size_t)ctx_->sm_count * 2));
        if (blocks < 1) blocks = 1;
        HG_K(ctx_, KC_DOT, (size_t)ntab * n * sizeof(T),
             k_dot_eq<FP, T><<<dim3(blocks, ntab), HG_BLOCK, 0, ctx_->stream>>>(tables, stride, n, lo, d_eq_.p, d_eq_.p + ((size_t)1 << lo), d_partials_.p, d_counters_.p, ch.d_msg(msg_off)));
    }
    template <class T> void eval_tables(Channel<FP>& ch, const T* tables, size_t stride, int ntab, size_t n, size_t point_idx, int nv, size_t msg_off) {
        build_eq(ch, point_idx, nv);
        dot_tables<T>(ch, tables, stride, ntab, n, msg_off);
    }

    // prove_grand_product (prover.rs:183-266) over nvec = 2m vectors of length N stored at tree (layer 0), upper layers appended
    // one grand product's tree and message slots: what build_tree_rest needs, and build_trees when the launches were deferred (prefetch mode)
    struct GpPlan { B* tree = nullptr; size_t N = 0; int nvars = 0; size_t roots_off = 0, ev0_off = 0, job_begin = 0; bool level1_done = false; };
    // does layer k of a tree over vectors of length N get its round 0 from a streaming kernel (tables longer than the tail kernel takes)?
    bool gp_needs_r0(size_t N, int k, int nvars) const { return k <= nvars - 2 && ((N >> k) / 2) > ((size_t)1 << FP::GP_TAIL_LOG); }
    // shared memory of k_gp_tail when a layer's 2m terms are split over `groups` CTAs: (1 + 2 tpg) tables of 2^GP_TAIL_LOG entries + half as many folded
    size_t gp_tail_smem(int groups) const {
        const int tpg = (2 * m_ + groups - 1) / groups;
        return ((size_t)(1 + 2 * tpg) * (((size_t)1 << FP::GP_TAIL_LOG) + ((size_t)1 << FP::GP_TAIL_LOG) / 2) + 32 * 4) * sizeof(X);
    }
    // position blocks per vector of the fused builders: every CTA ends with a block-level reduction that costs about as much as
    // one pass over its data, so CTAs are long (~16 per SM over the whole launch, at least 8 positions per thread)
    int fused_nxb(size_t work, int nvec) const {
        constexpr int ctas_per_sm = 16;
        const size_t by_work = (work + (size_t)HG_FUSED_BLOCK * 8 - 1) / ((size_t)HG_FUSED_BLOCK * 8);
        const size_t by_grid = std::max<size_t>(1, (size_t)ctx_->sm_count * ctas_per_sm / nvec);
        return (int)std::max<size_t>(1, std::min(by_work, by_grid));
    }
    X* r0_alloc(size_t nblk) {
        const size_t need = nblk * 4;
        if (r0_used_ + need > d_r0part_.n) throw std::runtime_error("LassoNode: round-0 partial pool too small");
        X* p = d_r0part_.p + r0_used_;
        r0_used_ += need;
        return p;
    }
    // one fused builder step of a tree (k_tree_up_r0): its arguments, whether it builds two levels, its grid and algorithmic bytes
    struct TreeStep { TreeR0Args<FP> a; bool two; unsigned nblk; size_t bytes; };
    // the fused steps of one tree (layers whose round 0 is streamed); *cur_out = last complete layer afterwards
    std::vector<TreeStep> plan_tree_fused(const GpPlan& pl, std::vector<GpLayerJob<FP>>& jobs, int* cur_out) {
        const int nvec = 2 * m_, nvars = pl.nvars;
        const size_t N = pl.N;
        std::vector<B*> layer(nvars);
        layer[0] = pl.tree;
        for (int k = 1; k < nvars; k++) layer[k] = layer[k - 1] + (size_t)nvec * (N >> (k - 1));
        auto job_of = [&](int k) -> GpLayerJob<FP>& { return jobs[pl.job_begin + (size_t)(nvars - 2 - k)]; };  // sumcheck nv = nvars-1-k is job nv-1
        int cur = pl.level1_done ? 1 : 0;  // last layer that is complete
        std::vector<TreeStep> steps;
        while (cur < nvars - 1 && gp_needs_r0(N, cur, nvars)) {
            const bool two = cur + 2 <= nvars - 1 && gp_needs_r0(N, cur + 1, nvars);
            const size_t len = N >> cur, q = two ? len / 4 : len / 2;
            TreeStep st;
            TreeR0Args<FP>& a = st.a;
            a.in = layer[cur]; a.out1 = layer[cur + 1]; a.out2 = two ? layer[cur + 2] : nullptr;
            a.q = q; a.nvec = nvec; a.own = own_range(nvec);
            a.nxb = fused_nxb(q / 2, nvec);
            const size_t nblk = (size_t)a.nxb * nvec;
            GpLayerJob<FP>& ja = job_of(cur);
            a.cA = ja.coef; a.partA = r0_alloc(nblk);
            ja.r0part = a.partA; ja.r0n = (int)nblk;
            a.cB = nullptr; a.partB = nullptr;
            if (two) {
                GpLayerJob<FP>& jb = job_of(cur + 1);
                a.cB = jb.coef; a.partB = r0_alloc(nblk);
                jb.r0part = a.partB; jb.r0n = (int)nblk;
            }
            st.two = two; st.nblk = (unsigned)nblk;
            st.bytes = (size_t)nvec * (len + len / 2 + (two ? len / 4 : 0)) * sizeof(B);  // the layer read once, the layer(s) above written once
            steps.push_back(st);
            cur += two ? 2 : 1;
        }
        *cur_out = cur;
        return steps;
    }
    void launch_tree_step(const TreeStep& x, const TreeStep* y) {  // y: the step of the other tree that shares the launch (same `two`), or nullptr
        cudaStream_t s = ctx_->stream;
        KernelScope ks(ctx_, KC_TREE, x.bytes + (y ? y->bytes : 0));
        const unsigned grid = x.nblk + (y ? y->nblk : 0);
        if (x.two) k_tree_up_r0<FP, true><<<grid, HG_FUSED_BLOCK, 0, s>>>(x.a, y ? y->a : x.a, x.nblk);
        else k_tree_up_r0<FP, false><<<grid, HG_FUSED_BLOCK, 0, s>>>(x.a, y ? y->a : x.a, x.nblk);
        HG_LAUNCH_CHECK();
    }
    // both product trees of the node (prover.rs:191-195, Layer::up :332-354). The builders also sample round 0 of every layer that
    // is streamed (gp_fused.cuh) and the layer jobs get the partial-sum regions; step k of both trees shares a launch.
    void build_trees(Channel<FP>& ch, const GpPlan& pl1, const GpPlan& pl2, std::vector<GpLayerJob<FP>>& jobs) {
        int cur1 = 0, cur2 = 0;
        const std::vector<TreeStep> s1 = plan_tree_fused(pl1, jobs, &cur1), s2 = plan_tree_fused(pl2, jobs, &cur2);
        size_t k2 = 0;
        for (size_t k1 = 0; k1 < s1.size(); k1++) {
            const TreeStep* mate = (k2 < s2.size() && s2[k2].two == s1[k1].two) ? &s2[k2] : nullptr;
            launch_tree_step(s1[k1], mate);
            if (mate) k2++;
        }
        for (; k2 < s2.size(); k2++) launch_tree_step(s2[k2], nullptr);
        build_tree_rest(ch, pl1, cur1);
        build_tree_rest(ch, pl2, cur2);
    }
    // the levels above the fused part of one tree and its top
    void build_tree_rest(Channel<FP>& ch, const GpPlan& pl, int cur) {
        cudaStream_t s = ctx_->stream;
        const int nvec = 2 * m_, nvars = pl.nvars;
        const size_t N = pl.N;
        std::vector<B*> layer(nvars);
        layer[0] = pl.tree;
        for (int k = 1; k < nvars; k++) layer[k] = layer[k - 1] + (size_t)nvec * (N >> (k - 1));
        for (int k = cur + 1; k < nvars;) {
            const size_t len_prev = N >> (k - 1);  // vector length of the layer this step reads
            if (len_prev <= (size_t)HG_TREE_TAIL && len_prev > 2) {  // the rest of the tree in one launch (shared memory)
                HG_K(ctx_, KC_TREE, (size_t)nvec * len_prev * 2 * sizeof(B),
                     k_tree_tail<FP><<<nvec, 256, len_prev * sizeof(B), s>>>(layer[k - 1], nvec, (int)len_prev, own_range(nvec)));
                break;
            }
            if (k + 1 < nvars) {  // two levels per launch: layer k is written and never re-read by the build
                const size_t q = N >> (k + 1);
                HG_K(ctx_, KC_TREE, (size_t)nvec * q * 7 * sizeof(B),
                     k_tree_up2<FP><<<dim3((unsigned)(((q >= 2 ? q / 2 : q) + HG_BLOCK - 1) / HG_BLOCK), nvec), HG_BLOCK, 0, s>>>(layer[k - 1], layer[k], layer[k + 1], q, own_range(nvec)));
                k += 2;
            } else {
                const size_t h = N >> k;
                HG_K(ctx_, KC_TREE, (size_t)nvec * h * 3 * sizeof(B), k_tree_up<FP><<<dim3((unsigned)((h + HG_BLOCK - 1) / HG_BLOCK), nvec), HG_BLOCK, 0, s>>>(layer[k - 1], layer[k], h, own_range(nvec)));
                k += 1;
            }
        }
        HG_K(ctx_, KC_TREE, (size_t)nvec * 2 * sizeof(B), k_tree_top<FP><<<(nvec + HG_BLOCK - 1) / HG_BLOCK, HG_BLOCK, 0, s>>>(layer[nvars - 1], own_begin(nvec), own_end(nvec), ch.d_msg(pl.roots_off), ch.d_msg(pl.ev0_off)));
    }

    void grand_product(Channel<FP>& ch, const WireOptions& wo, B* tree, size_t N, size_t* point_idx, std::vector<GpLayerJob<FP>>* batch,
                       bool level1_done, GpPlan* defer = nullptr) {
        const int nvec = 2 * m_;
        int nvars = 0;
        while (((size_t)1 << nvars) < N) nvars++;
        // layer k has vectors of length N >> k, k = 0..nvars-1 (prover.rs:191-195)
        std::vector<B*> layer(nvars);
        layer[0] = tree;
        for (int k = 1; k < nvars; k++) layer[k] = layer[k - 1] + (size_t)nvec * (N >> (k - 1));
        const size_t roots_off = ch.alloc_msg(nvec), ev0_off = ch.alloc_msg(2 * nvec);
        GpPlan pl;
        pl.tree = tree; pl.N = N; pl.nvars = nvars; pl.level1_done = level1_done; pl.job_begin = batch ? batch->size() : 0;
        pl.roots_off = roots_off; pl.ev0_off = ev0_off;
        if (defer) *defer = pl;
        else build_tree_rest(ch, pl, level1_done ? 1 : 0);
        struct GpHost { std::vector<X> claimed; std::vector<X> evals; size_t mu_idx = 0; bool pending = false; };
        auto gp = std::make_shared<GpHost>();
        Channel<FP>* chp = &ch;
        ch.emit([chp, gp, roots_off, ev0_off, nvec]() {
            auto& t = chp->transcript();
            gp->claimed.resize(nvec);
            for (int i = 0; i < nvec; i++) { gp->claimed[i] = chp->msg(roots_off + i); t.write_felt_ext(gp->claimed[i]); }  // prover.rs:197-221
            gp->evals.resize(2 * nvec);
            for (int i = 0; i < 2 * nvec; i++) { gp->evals[i] = chp->msg(ev0_off + i); t.write_felt_ext(gp->evals[i]); }   // prover.rs:257
        });
        size_t mu_idx = ch.squeeze(1);  // prover.rs:259
        size_t first_chal = mu_idx;
        for (int nv = 1; nv < nvars; nv++) {
            const size_t prev_mu = mu_idx;
            const size_t gamma_idx = ch.squeeze(1);  // prover.rs:238
            auto st = std::make_shared<ScHostState<FP>>();
            const int asc = wo.a5_ascending;
            ch.emit([chp, gp, st, prev_mu, gamma_idx, nvec, asc]() {
                // layer_down_claim (prover.rs:288-294) then sum_check_claim (prover.rs:281-286)
                X mu = chp->chal(prev_mu), g = chp->chal(gamma_idx);
                X claim = FP::x_zero(), p = FP::x_one();
                for (int i = 0; i < nvec; i++) {
                    X l = gp->evals[2 * i], r = gp->evals[2 * i + 1];
                    gp->claimed[i] = FP::x_add(l, FP::x_mul(mu, FP::x_sub(r, l)));
                    claim = FP::x_add(claim, FP::x_mul(gp->claimed[i], p));
                    p = FP::x_mul(p, g);
                }
                (void)asc;  // the claim always uses ascending powers (prover.rs:281-286); only the expression order is an assumption
                st->claim = claim;
            });
            size_t sc_first = 0, ev_off = 0;
            bool scaled = false;
            const B* tables = layer[nvars - 1 - nv];
            gp_sumcheck_dev<FP>(ctx_, ch, wo, tables, (size_t)1 << nv, nvec, ch.d_chal(gamma_idx), d_gp_coeffs_.p, d_bufA_.p, d_bufB_.p, sc_, st, &sc_first, &ev_off, &scaled, batch, gamma_idx);
            ch.emit([chp, gp, ev_off, nvec, scaled, gamma_idx, asc]() {
                auto& t = chp->transcript();
                // the device keeps l_i (i > 0) and r_0 pre-multiplied by c_i (gp_kernels.cuh); undo it exactly with c_i^{-1}
                X ginv = FP::x_inv(chp->chal(gamma_idx)), p = FP::x_one();
                std::vector<X> cinv(nvec);
                for (int i = 0; i < nvec; i++) { cinv[asc ? i : nvec - 1 - i] = p; p = FP::x_mul(p, ginv); }
                for (int i = 0; i < 2 * nvec; i++) {
                    X e = chp->msg(ev_off + i);
                    if (scaled && (i == 1 || ((i & 1) == 0 && i > 0))) e = FP::x_mul(e, cinv[i / 2]);  // c_i sits on l_i (i > 0) and on r_0
                    gp->evals[i] = e;
                    t.write_felt_ext(e);  // prover.rs:257
                }
            });
            mu_idx = ch.squeeze(1);
            first_chal = sc_first;
        }
        // x = round challenges of the bottom layer ++ [mu]  (prover.rs:261-264): contiguous in squeeze order
        if (nvars > 1 && mu_idx != first_chal + (size_t)(nvars - 1)) throw std::runtime_error("grand_product: challenge layout broken");
        *point_idx = first_chal;
    }

    // all layer sumchecks of both grand products, batched: round j of every layer in one launch, then one tail launch
    // coefficient tables [c_i | c_i r_0] of every layer of both grand products, one launch (needs only challenges)
    void prepare_gp_coeffs(Channel<FP>& ch, const WireOptions& wo, std::vector<GpLayerJob<FP>>& jobs) {
        cudaStream_t s = ctx_->stream;
        const int nl = (int)jobs.size();
        r0_used_ = 0;
        if (!nl) return;
        size_t coef_off = 0;
        std::vector<GpCoeffItem<FP>> citems(nl);
        for (int k = 0; k < nl; k++) {
            auto& j = jobs[k];
            j.coef = d_gp_coeffs_.p + coef_off;
            coef_off += 2 * (size_t)j.nvec;
            citems[k].gamma = ch.d_chal(j.gamma_idx);
            citems[k].r0 = j.nv >= 2 ? ch.d_chal(j.r0_idx) : nullptr;
            citems[k].c = j.coef; citems[k].cr = j.coef + j.nvec; citems[k].n = j.nvec;
        }
        if (coef_off > d_gp_coeffs_.n) throw std::runtime_error("prepare_gp_coeffs: pool too small");
        const size_t bytes = citems.size() * sizeof(GpCoeffItem<FP>);
        if (h_cdesc_.n < bytes) { h_cdesc_.alloc(bytes * 2); d_cdesc_.alloc(bytes * 2); }
        memcpy(h_cdesc_.p, citems.data(), bytes);
        HG_CUDA(cudaMemcpyAsync(d_cdesc_.p, h_cdesc_.p, bytes, cudaMemcpyHostToDevice, s));
        HG_K(ctx_, KC_MISC, 0, k_gp_coeffs_multi<FP><<<nl, 64, 0, s>>>((const GpCoeffItem<FP>*)d_cdesc_.p, wo.a5_ascending));
    }

    void run_gp_batch(Channel<FP>& ch, const WireOptions& wo, const std::vector<GpLayerJob<FP>>& jobs) {
        cudaStream_t s = ctx_->stream;
        const int nl = (int)jobs.size();
        if (!nl) return;
        (void)wo;
        constexpr size_t tail_n = (size_t)1 << FP::GP_TAIL_LOG;
        // Round r of a streamed layer samples h_r on the level-r tables L_r (|L_r| = n >> r). All challenges are on the device, so
        // every round writes its tables folded by its own challenge, L_{r+1}, and the next round reads those pairs: round 1 reads
        // the base tables L_0 (folding by r_0 on read, scaling by c_i) and writes L_2, round r >= 2 reads L_r and writes L_{r+1}.
        // carve per-layer regions out of the pools: odd rounds write bufA, even rounds bufB
        std::vector<X*> bufA(nl, nullptr), bufB(nl, nullptr), coef(nl, nullptr);
        size_t pool_off = 0;
        for (int k = 0; k < nl; k++) {
            const auto& j = jobs[k];
            coef[k] = j.coef;
            if (j.n > tail_n) {
                size_t a = 2 * (size_t)j.nvec * (j.n / 4), b = 2 * (size_t)j.nvec * (j.n / 8);
                bufA[k] = d_pool_.p + pool_off; pool_off += a;
                bufB[k] = d_pool_.p + pool_off; pool_off += b;
            }
        }
        if (pool_off > d_pool_.n) throw std::runtime_error("run_gp_batch: pool too small");
        // Rounds of layer k: round 0 sampled by the fused tree builders, streamed launches r = 1..S_k, then the tail kernel from
        // 2^GP_TAIL_LOG entries on. Round 1 is always streamed: it scales the tables by c_i. S_k = 0: the whole layer runs in the tail.
        std::vector<int> S(nl, 0);
        int maxJ = 0;
        for (int k = 0; k < nl; k++) {
            const auto& j = jobs[k];
            if (j.n <= tail_n) continue;
            if (j.r0n == 0) throw std::runtime_error("run_gp_batch: a streamed layer has no round 0 from the tree builders");
            S[k] = j.nv - FP::GP_TAIL_LOG;
            maxJ = std::max(maxJ, S[k]);
        }
        std::vector<std::vector<GpItem<FP>>> rounds(maxJ + 1);  // indexed by round; rounds[0] stays empty
        std::vector<size_t> round_bytes(maxJ + 1, 0);
        size_t part_need = 0;
        // grid shape of the streaming launches: at most max_bx_per_sm blocks per SM along a table, term groups added until an item
        // has about FP::GP_TARGET blocks (in units of the SM count)
        constexpr int max_bx_per_sm = 4;
        // measured optimum: one term group (every thread loops over all terms of its pairs and reuses t_0) as soon as a table gives
        // ~37 CTAs; smaller layers get term groups so that no layer runs on fewer CTAs than that
        const int target_blocks = std::max(1, (int)(ctx_->sm_count * FP::GP_TARGET * (HG_BLOCK / FP::GP_BLOCK)));
        const size_t gp_max_bx = (size_t)ctx_->sm_count * max_bx_per_sm * (HG_BLOCK / FP::GP_BLOCK);
        // Work-balanced shape (fields with FP::GP_BALANCE): a round finishes with its slowest CTA, and a CTA's time is (terms it
        // loops over) x (positions per thread). With one term group per large layer the late rounds ran ~1000 CTAs of which the
        // largest layer's looped over all 2m terms while the SMs were half empty (profiles/r2_launch_list.md: round 5 93 us for
        // 0.3 GB). Here every item gets term groups of about total thread-terms / resident threads, so that the whole round is one
        // wave of equal CTAs, and the items are placed in the grid heaviest CTA first.
        constexpr int min_tpg = 4;
        const size_t resident_threads = (size_t)ctx_->sm_count * FP::GP_MIN_BLOCKS * HG_BLOCK;
        for (int r = 1; r <= maxJ; r++) {
            int blk = 0;
            size_t part_off = 0;
            // layers that take part in this round, their thread count along the table, and the round's total thread-terms
            std::vector<int> order;
            std::vector<size_t> tx(nl, 0);
            size_t total_tt = 0;
            for (int k = 0; k < nl; k++) {
                const auto& j = jobs[k];
                if (r > S[k]) continue;
                tx[k] = j.n >> (r + 1);  // pairs of L_r
                total_tt += std::min(tx[k], gp_max_bx * FP::GP_BLOCK) * (size_t)(own_end(j.nvec) - own_begin(j.nvec));
                order.push_back(k);
            }
            const size_t tpg_bal = std::max<size_t>((size_t)min_tpg, (total_tt + resident_threads - 1) / resident_threads);
            if (FP::GP_BALANCE)  // heaviest CTAs first: longer table (more positions per thread, the same term count) first
                std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return tx[a] > tx[b]; });
            for (int k : order) {
                const auto& j = jobs[k];
                GpItem<FP> it;
                it.nvec = j.nvec;
                it.i_begin = own_begin(j.nvec); it.i_end = own_end(j.nvec); it.write_t0 = it.i_begin > 0;
                const int nown = it.i_end - it.i_begin;
                it.c = coef[k]; it.cr = coef[k] + j.nvec;
                it.n_in = j.n >> (r == 1 ? 0 : r);
                it.in = (r == 1) ? (const void*)j.tables : (const void*)(((r - 1) & 1) ? bufA[k] : bufB[k]);
                it.out = (r & 1) ? bufA[k] : bufB[k];
                it.r_prev = ch.d_chal(j.r0_idx + r - 1);
                it.r_cur = ch.d_chal(j.r0_idx + r);
                it.msg = ch.d_msg(j.msg_off + 4 + 3 * (size_t)(r - 1));
                round_bytes[r] += (size_t)(2 * nown + it.write_t0) * (it.n_in * (r == 1 ? sizeof(B) : sizeof(X)) + (j.n >> (r + 1)) * sizeof(X));
                size_t b = (tx[k] + FP::GP_BLOCK - 1) / FP::GP_BLOCK;
                if (b < 1) b = 1;
                if (b > gp_max_bx) b = gp_max_bx;
                int g = (int)std::min<size_t>((size_t)nown, std::max<size_t>(1, ((size_t)target_blocks + b - 1) / b));
                if (FP::GP_BALANCE && tpg_bal * 5 < (size_t)nown * 4)  // (a split that saves less than a fifth of the loop is not worth re-folding t_0)
                    g = std::max(g, (int)std::max<size_t>(1, (size_t)nown / tpg_bal));  // rounded down: rather one wave of slightly longer CTAs than a second wave
                it.tpg = (nown + g - 1) / g;
                it.groups = (nown + it.tpg - 1) / it.tpg;
                it.bx = (int)b;
                it.nblk = it.bx * it.groups;
                it.blk_start = blk;
                blk += it.nblk;
                it.partials = d_gp_partials_.p + part_off;
                part_off += (size_t)it.nblk * 4;
                it.counter = d_gp_counters_.p + rounds[r].size();
                rounds[r].push_back(it);
            }
            part_need = std::max(part_need, part_off);
            if (rounds[r].size() > d_gp_counters_.n) throw std::runtime_error("run_gp_batch: too many layers");
        }
        if (part_need > d_gp_partials_.n) { d_gp_partials_.alloc(part_need * 2); /* re-point */
            for (auto& rv : rounds) { size_t off = 0; for (auto& it : rv) { it.partials = d_gp_partials_.p + off; off += (size_t)it.nblk * 4; } } }
        std::vector<GpTailItem<FP>> titems(nl);
        size_t tail_bytes = 0;
        for (int k = 0; k < nl; k++) {
            const auto& j = jobs[k];
            GpTailItem<FP>& t = titems[k];
            {
                const int nown = own_end(j.nvec) - own_begin(j.nvec);
                t.tpg = std::max(1, (j.nvec + tail_groups_ - 1) / tail_groups_);  // sized for all 2m terms: the shared-memory budget was checked for that
                t.groups = std::max(1, (nown + t.tpg - 1) / t.tpg);
                if ((size_t)k >= d_gp_tailcnt_.n) throw std::runtime_error("run_gp_batch: too many layers for the tail scratch");
                t.gpart = d_gp_tailpart_.p + (size_t)k * tail_groups_ * (HG_GP_TAIL_MAXR + 1) * 4;
                t.counter = d_gp_tailcnt_.p + k;
            }
            t.c = coef[k]; t.nvec = j.nvec; t.evals = ch.d_msg(j.evals_off);
            t.i_begin = own_begin(j.nvec); t.i_end = own_end(j.nvec);
            t.r0part = j.r0part; t.r0n = j.r0n;
            if (j.n <= tail_n) {
                t.from_base = 1; t.in = j.tables; t.n = (int)j.n; t.rounds = j.nv - 1;
                t.chal = ch.d_chal(j.r0_idx); t.msg0 = ch.d_msg(j.msg_off); t.msg = ch.d_msg(j.msg_off + 4);
                tail_bytes += 2 * (size_t)j.nvec * j.n * sizeof(B);
            } else {  // the tables the last streamed round wrote, L_{S+1}: the tail samples round S+1 on them, then folds by r_{S+1}, ...
                t.from_base = 0; t.in = (S[k] & 1) ? bufA[k] : bufB[k]; t.n = (int)(tail_n / 2); t.rounds = FP::GP_TAIL_LOG - 2;
                t.chal = ch.d_chal(j.r0_idx + S[k] + 1); t.msg0 = ch.d_msg(j.msg_off); t.msg = ch.d_msg(j.msg_off + 4 + 3 * (size_t)S[k]);
                tail_bytes += 2 * (size_t)j.nvec * t.n * sizeof(X);
            }
        }
        // upload descriptors
        size_t bytes = titems.size() * sizeof(GpTailItem<FP>) + 16;
        for (auto& rv : rounds) bytes += rv.size() * sizeof(GpItem<FP>) + 16;
        if (h_desc_.n < bytes) { h_desc_.alloc(bytes * 2); d_desc_.alloc(bytes * 2); }
        unsigned char* hp = h_desc_.p;
        size_t off = 0;
        auto put = [&](const void* src, size_t n) { size_t o = off; memcpy(hp + off, src, n); off += (n + 15) & ~(size_t)15; return o; };
        std::vector<size_t> r_off(rounds.size());
        for (size_t r = 0; r < rounds.size(); r++) r_off[r] = put(rounds[r].data(), rounds[r].size() * sizeof(GpItem<FP>));
        size_t t_off = put(titems.data(), titems.size() * sizeof(GpTailItem<FP>));
        if (off > h_desc_.n) throw std::runtime_error("run_gp_batch: descriptor staging overflow");
        HG_CUDA(cudaMemcpyAsync(d_desc_.p, h_desc_.p, off, cudaMemcpyHostToDevice, s));
        // launches
        for (size_t r = 1; r < rounds.size(); r++) {
            const auto& last = rounds[r].back();
            const int grid = last.blk_start + last.nblk, ni = (int)rounds[r].size();
            const GpItem<FP>* di = (const GpItem<FP>*)(d_desc_.p + r_off[r]);
            KernelScope ks(ctx_, KC_SC_GP, round_bytes[r]);
            if (r == 1) k_gp_fold_multi<FP, B, true><<<grid, FP::GP_BLOCK, 0, s>>>(di, ni);
            else k_gp_fold_multi<FP, X, false><<<grid, FP::GP_BLOCK, 0, s>>>(di, ni);
            HG_LAUNCH_CHECK();
        }
        {
            const size_t smem = gp_tail_smem(tail_groups_);
            KernelScope ks(ctx_, KC_SC_GP, tail_bytes);
            k_gp_tail<FP><<<nl * tail_groups_, HG_TAIL_THREADS, smem, s>>>((const GpTailItem<FP>*)(d_desc_.p + t_off), tail_groups_);
            HG_LAUNCH_CHECK();
        }
    }

    // device that opens read_ts / final_cts of chunk slot q: the owner of the slot's first read vector
    int slot_owner(int q) const {
        const int nvec = 2 * m_;
        for (int pos = 0; pos < m_; pos++)
            if (pos_slot_host_[pos] == q)
                for (int r = 0; r < shard_world_; r++)
                    if (pos >= (int)((size_t)nvec * r / shard_world_) && pos < (int)((size_t)nvec * (r + 1) / shard_world_)) return r;
        return 0;
    }
    // does this device read the access counters of chunk slot q? (hashes of its own vectors and of vector 0, its counter openings)
    bool slot_needed(int q) const {
        if (shard_world_ == 1) return true;
        if (pos_slot_host_[0] == q || slot_owner(q) == shard_rank_) return true;
        for (int v = own_begin(2 * m_); v < own_end(2 * m_); v++) if (pos_slot_host_[v % m_] == q) return true;
        return false;
    }
    // vectors [own_begin, own_end) of a grand product belong to this device (all of them unless prove_shard is running)
    VecRange own_range(int nvec) const { VecRange r; r.lo = own_begin(nvec); r.hi = own_end(nvec); return r; }
    int own_begin(int nvec) const { return (int)((size_t)nvec * shard_rank_ / shard_world_); }
    int own_end(int nvec) const { return (int)((size_t)nvec * (shard_rank_ + 1) / shard_world_); }
    int shard_rank_ = 0, shard_world_ = 1;
    size_t shard_r_idx_ = 0, shard_sum_off_ = 0;
    double timing_[4] = {0, 0, 0, 0};
    size_t msg_budget_ = 0;
    int eq_nv_ = 0;
    DeviceCtx* ctx_;
    LassoPreprocessing pp_;
    int num_vars_, log2M_ = 16, m_ = 0, nslots_ = 0, rows_per_block_ = 4096, nblk_cnt_ = 1, max_blocks_ = 0;
    size_t n_rows_, R_ = 0, M_ = 0, total_chal_ = 0;
    NodeMeta meta_host_;
    std::vector<int> chunk_dims_;
    std::vector<std::vector<int>> chunk_mems_;
    std::vector<u64> slot_used_;
    std::vector<int> pos_slot_host_;  // chunk slot of the memory at chunk-major position pos
    std::vector<int> slot_addr_dim_;
    std::vector<B> coll_coeff_host_;
    DevBuf<NodeMeta> d_meta_;
    DevBuf<u8> d_row_lookup_;
    DevBuf<B> d_subtables_, d_E_, d_coll_, d_out_, d_coeff_coll_, d_wpow_, d_tree1_, d_tree2_;
    DevBuf<u16> d_dims_;
    DevBuf<u32> d_read_cts_, d_final_cts_, d_cnt_hist_, d_cnt_misc_, d_cnt_runs_;
    DevBuf<u64> d_cnt_a_, d_cnt_b_;
    size_t cnt_cap_ = 0;
    DevBuf<int> d_pos_mem_, d_pos_dim_, d_pos_slot_, d_pos_sub_;
    DevBuf<X> d_eq_, d_gp_coeffs_, d_bufA_, d_bufB_, d_partials_, d_coll_terms_;
    int coll_coeff_state_ = 0;  // 0 not uploaded, 1 ascending, 2 descending
    DevBuf<unsigned> d_counters_, d_gp_counters_;
    DevBuf<X> d_pool_, d_gp_partials_, d_r0part_, d_midpart_, d_gp_tailpart_;
    DevBuf<unsigned> d_gp_tailcnt_;
    int tail_groups_ = 1;
    size_t r0_used_ = 0;
    DevBuf<unsigned char> d_desc_, d_cdesc_;
    PinnedBuf<unsigned char> h_desc_, h_cdesc_;
    ScScratch sc_;
    std::unique_ptr<Channel<FP>> ch_;
};

}  // namespace hg
