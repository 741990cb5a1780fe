// Host-side runner of the four-step NTT (ntt.cuh) with a per-size twiddle cache.
#pragma once
#include <map>
#include <memory>

#include "ntt.cuh"
#include "prover.cuh"

namespace hg {

template <class FP> class NttEngine {
  public:
    typedef typename FP::B B;
    explicit NttEngine(DeviceCtx* ctx) : ctx_(ctx) {}
    // batched in-place transform of `batch` consecutive vectors of 2^log_n base elements at d_data (device)
    void run(B* d_data, int log_n, bool inverse, size_t batch) {
        if (log_n < 1 || log_n > 24 || log_n > FP::TWO_ADICITY) throw std::runtime_error("hg_ntt: log_n out of range");
        cudaStream_t s = ctx_->stream;
        const size_t N = (size_t)1 << log_n;
        const int key = log_n * 2 + (inverse ? 1 : 0);
        auto& tw = twiddles_[key];
        if (!tw) {
            tw.reset(new DevBuf<B>());
            tw->alloc(N);
            HG_K(ctx_, KC_MISC, N * sizeof(B), k_ntt_twiddles<FP><<<(unsigned)((N + 255) / 256), 256, 0, s>>>(log_n, inverse ? 1 : 0, FP::root_of_unity(), tw->p));
        }
        if (scratch_.n < N * batch) { HG_CUDA(cudaStreamSynchronize(s)); scratch_.alloc(N * batch); }
        const int log_n1 = (log_n + 1) / 2, log_n2 = log_n - log_n1;
        const int n1 = 1 << log_n1, n2 = 1 << log_n2;
        const int tile_c = std::min(HG_NTT_TILE, n2), tile_r = std::min(HG_NTT_TILE, n1);
        // data tile + the n/2 twiddles of the in-tile transform
        const size_t smem_c = ((size_t)n1 * (tile_c | 1) + n1 / 2 + 1) * sizeof(B), smem_r = ((size_t)n2 * (tile_r | 1) + n2 / 2 + 1) * sizeof(B);
        if (smem_c > 200 * 1024 || smem_r > 200 * 1024) throw std::runtime_error("hg_ntt: transform too large for the shared-memory tiles");
        HG_K(ctx_, KC_NTT, 2 * N * batch * sizeof(B),
             k_ntt_cols<FP><<<dim3(n2 / tile_c, (unsigned)batch), HG_NTT_THREADS, smem_c, s>>>(d_data, scratch_.p, log_n1, log_n2, tile_c, tw->p));
        const B scale = inverse ? FP::b_inv(FP::b_from_u64(N)) : FP::b_one();
        HG_K(ctx_, KC_NTT, 2 * N * batch * sizeof(B),
             k_ntt_rows<FP><<<dim3(n1 / tile_r, (unsigned)batch), HG_NTT_THREADS, smem_r, s>>>(scratch_.p, d_data, log_n1, log_n2, tile_r, tw->p, scale, inverse ? 1 : 0));
    }

  private:
    DeviceCtx* ctx_;
    std::map<int, std::unique_ptr<DevBuf<B>>> twiddles_;
    DevBuf<B> scratch_;
};

}  // namespace hg
