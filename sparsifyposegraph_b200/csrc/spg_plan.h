// spg_plan.h — kernel parameter block and shared-memory plan of blanket_kernel (host + device).
#pragma once
#include <cstdint>

#include "../../include/spg_capi.h"
#include "../../include/spg_record.h"
#include "spg_device.cuh"

namespace spg {

// shared-memory plan of fast_kernel (spg_fast.cuh), in doubles; computed on the host by fast_plan<D>()
struct FastPlan {
    int NP, ntiles, chunk;
    int off_pose, off_B, off_P, off_W, off_small, off_U, total;
    int off_h00, off_hk0, off_y, off_jm; // phase A inside the union region U (after the record copy)
    int off_set2; // C and G sweeps side by side: second panel set at off_B + off_set2 (0: one sweep after the other)
};

struct KernelParams {
    int32_t algorithm, topology;
    double chord_ratio;
    int32_t flags;               // bit 0: force the general (eigen-decomposition) NFR path
    int32_t lean;                // buf2 holds sweep / J Sigma scratch only (NFR rounds of POSE edges): two CTAs per SM
    int32_t n_list;              // blankets handled by this launch
    const int32_t *list;         // their indices (NULL: identity)
    const int64_t *rec_off;
    const uint64_t *records;
    const int64_t *out_off;
    uint64_t *out;
    double *dbg_target;
    const int64_t *dbg_target_off;
    double *dbg_weights;
    const int64_t *dbg_weights_off;
    // shared-memory carve-up of this bucket (all in doubles)
    int32_t max_nv, max_e, max_rec_words;
    int32_t off_pose, off_buf0, off_buf1, off_buf2, off_small, total_doubles;
    int32_t buf0_doubles, buf1_doubles, buf2_doubles;
    int32_t off_glc, glc_doubles; // GLC scratch (only for algorithm == SPG_ALG_GLC launches)
    int32_t glc_warps;            // GLC tree: warps that finish factors side by side (0: plan_smem picks by CTA width)
    int32_t glc_warp_doubles;     // scratch of one such warp
    double *nfr_ws;               // per-CTA workspace of the iterative NFR fit (global memory)
    int64_t nfr_ws_stride;        // doubles per CTA
    double *gws;                  // spill variant: per-CTA slice holding the whole buffer plan (global memory)
    int64_t gws_stride;           // doubles per CTA
    unsigned long long *prof;     // optional: 16 per-stage cycle accumulators (thread 0 of every CTA)
    // fast_kernel (spg_fast.cuh) appends the blankets it does not take to retry_list (atomic counter retry_count);
    // the follow-up blanket_kernel launch reads its blanket count from n_list_dev (= retry_count) instead of n_list
    int32_t *retry_list;
    int32_t *retry_count;
    const int32_t *n_list_dev;
    FastPlan fast;
};

constexpr int ASM_CHUNK = 8; // edges linearised per pre-pass

// Host-side: shared-memory layout for a bucket with at most max_nv vertices (n_removed >= 1),
// max_e edges and max_rec_words record words.
template <int D>
inline void plan_smem(KernelParams &p) {
    const int PS = PoseStride<D>::value;
    const int N = D * p.max_nv;
    const int kmax = D * (p.max_nv - 1);
    const int nk = p.max_nv - 1;
    const int pairs = nk * (nk - 1) / 2;
    int o = p.max_rec_words > 400 ? p.max_rec_words : 400; // record copy; after the assembly: pivot columns of two concurrent sweeps
    p.off_pose = o;  o += p.max_nv * PS;
    p.off_buf0 = o;
    p.buf0_doubles = N * odd_ld(N);
    o += p.buf0_doubles;
    p.off_buf1 = o;
    int b1 = kmax * odd_ld(kmax > 0 ? kmax : 1);
    int asm_scratch = ASM_CHUNK * 2 * (D * 2 * D);
    const int sweep_scratch = 392; // pivot-column buffers of the register-tiled sweeps (2 parities x 2 columns x 96 + pad; buf1 or buf2)
    p.buf1_doubles = b1 > asm_scratch ? b1 : asm_scratch;
    if(p.buf1_doubles < sweep_scratch) p.buf1_doubles = sweep_scratch;
    o += p.buf1_doubles;
    p.off_buf2 = o;
    p.buf2_doubles = (nk >= 2) ? (b1 > sweep_scratch ? b1 : sweep_scratch) : 0; // eigenvectors / sweep scratch
    if(p.lean) { // pivot columns of a sweep (392) or Tm = J Sigma of the closed form (one D x 2D block per tree edge)
        const int tm = nk * D * 2 * D;
        p.buf2_doubles = tm > 400 ? tm : 400;
    }
    o += p.buf2_doubles;
    p.off_small = o;
    // small: w[kmax] order[kmax](int) cs[kmax+2] red[34] weights[pairs] heapw[pairs] heapab[pairs] (int2)
    //        tree[2*max(pairs,1)] (int) uf[nk] (int) Lfac[nk*D*D] logd[nk] misc[16]
    o += kmax + (kmax + 1) / 2 + (kmax + kmax / 2 + 4) + 34 + pairs + pairs + pairs + (pairs > 0 ? pairs : 1) + (nk + 1) / 2 + 1 +
         nk * D * D + nk + 16;
    p.off_glc = o;
    p.glc_doubles = 0;
    if(p.algorithm == SPG_ALG_GLC) {
        // tree: joint (4D^2) + target (4D^2) + pinv out (D^2) + pinv scratch + getEdge scratch (c = 2D);
        // dense: meas k + blocks 2 nk D^2 + Jacobi scratch + order
        const int c = 2 * D;
        // per warp: joint (4D^2) + target (4D^2) + pinv out (D^2) + pinv scratch + getEdge scratch (c = 2D) + vertex pair
        p.glc_warp_doubles = 4 * D * D + 4 * D * D + D * D + (2 * D * (D | 1) + 2 * D + 16) + (8 * c * c + 8 * c + 64) + 2;
        if(p.glc_warps <= 0) { // warps of the CTA width launch_general picks for this N, at most 4
            const int NN = D * p.max_nv;
            p.glc_warps = NN <= 12 ? 1 : (NN <= 32 ? 2 : 4);
        }
        const int tree = p.glc_warps * p.glc_warp_doubles;
        // dense: meas k + blocks 2 nk D^2 + Jacobi scratch + order
        const int dense = kmax + 2 * nk * D * D + (kmax + kmax / 2 + 8) + 8 + kmax / 2 + 2;
        p.glc_doubles = (tree > dense ? tree : dense) + 8;
        o += p.glc_doubles;
    }
    p.total_doubles = o;
}

} // namespace spg
