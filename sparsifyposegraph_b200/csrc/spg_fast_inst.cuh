// spg_fast_inst.cuh — launch wrapper of one fast_kernel<D, G, MAXW> instantiation (spg_fast.cuh).
#pragma once
#include <algorithm>
#include <cstdlib>
#include <mutex>

#include "spg_ctx.h"
#include "spg_fast.cuh"

namespace {
// G = 8 / 16 / 32: sub-warp groups, 32 / G blankets per warp, up to MAXW such warps per CTA (phase barriers keep them in
// the same stage, see SPG_PHASE in spg_fast.cuh); G = 0: one blanket per CTA of up to MAXW warps.
// Returns SPG_ERR_UNSUPPORTED when the bucket does not fit this instantiation (the caller runs blanket_kernel alone).
template <int D, int G, int MAXW>
spg_status launch_fast(spg_ctx *ctx, spg::KernelParams &kp) {
    static std::mutex mu;
    static bool configured[64] = {};
    constexpr int SPW = G ? 32 / (G ? G : 1) : 1; // blanket slots per warp
    // shared memory per blanket slot that still lets the register file's warp / CTA count (MINB) be resident
    constexpr int MINB = G ? (D == 6 ? 12 : 16) : (MAXW <= 4 ? 3 : (D == 6 ? 1 : 2));
    const size_t budget = std::min<size_t>(ctx->smem_optin, (size_t) (228 * 1024) / MINB - 1024) / SPW;
    // CTA-wide kernels sweep C and the anchored G side by side (one thread per block of either, nk^2 threads) when the
    // CTA has room for them: half the serial block steps per blanket
    const int nk = kp.max_nv > 1 ? kp.max_nv - 1 : 1;
    const bool fused = G == 0 && nk * nk <= 32 * MAXW;
    const spg::FastPlan pl = spg::fast_plan<D>(kp.max_nv, kp.max_e, kp.max_rec_words, budget, fused);
    kp.fast = pl;
    const size_t warp_smem = (size_t) pl.total * SPW * sizeof(double);
    const int tiles = spg::fast_tiles(kp.max_nv);
    int warps = G ? 1 : ((fused ? nk * nk : tiles) + 31) / 32;
    if(warp_smem > ctx->smem_optin || warps > MAXW || (G && tiles > G)) return SPG_ERR_UNSUPPORTED;
    if(G) {
        // warps per CTA: a wide round gets as many as the registers (MAXW) and the shared memory allow, one CTA per SM;
        // a narrow round is spread over the SMs first (its latency is what the caller waits for)
        const int64_t need = ((int64_t) kp.n_list + SPW - 1) / SPW; // warps of work
        const int cap = (int) std::min<size_t>((size_t) MAXW, ctx->smem_optin / warp_smem);
        warps = (int) std::max<int64_t>(1, std::min<int64_t>(cap, (need + ctx->sm_count - 1) / ctx->sm_count));
        if(const char *e = getenv("SPG_FAST_WPC")) warps = std::max(1, std::min(cap, atoi(e))); // experiments
    }
    const int threads = 32 * warps;
    const size_t smem = G ? warp_smem * warps : warp_smem;
    {
        std::lock_guard<std::mutex> lk(mu);
        const int dv = ctx->device & 63;
        if(!configured[dv]) {
            SPG_CUDA(cudaFuncSetAttribute(spg::fast_kernel<D, G, MAXW>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) ctx->smem_optin));
            SPG_CUDA(cudaFuncSetAttribute(spg::fast_kernel<D, G, MAXW>, cudaFuncAttributePreferredSharedMemoryCarveout,
                                          (int) cudaSharedmemCarveoutMaxShared));
            configured[dv] = true;
        }
    }
    int per_sm = 0;
    SPG_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, spg::fast_kernel<D, G, MAXW>, threads, smem));
    if(per_sm < 1) return SPG_ERR_UNSUPPORTED;
    if(const char *e = getenv("SPG_FAST_CTAS")) per_sm = std::max(1, std::min(per_sm, atoi(e))); // experiments: resident CTAs per SM
    const int64_t per_cta = G ? (int64_t) SPW * warps : 1;
    const int64_t ctas = ((int64_t) kp.n_list + per_cta - 1) / per_cta;
    const int grid = (int) std::min<int64_t>(ctas, (int64_t) per_sm * ctx->sm_count);
    if(grid < 1) return SPG_OK;
    kp.prof = ctx->profiling ? reinterpret_cast<unsigned long long *>(ctx->d_prof.p) + 16 : nullptr;
    spg::fast_kernel<D, G, MAXW><<<grid, threads, smem, ctx->stream>>>(kp);
    SPG_CUDA(cudaGetLastError());
    ctx->launches++;
    ctx->fast_ctas_per_sm = per_sm;
    return SPG_OK;
}
} // namespace
