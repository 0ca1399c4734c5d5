// spg_capi.cu — C ABI of libspg_b200.so, blanket level (include/spg_capi.h).
// Host side of one wavefront round: bucket the blankets of the round by size, copy the packed
// records to HBM, launch one fused kernel per bucket (shared memory and CTA width sized to the
// bucket), copy the substitute-edge records back. No CPU fallback: without an sm_100 device every
// entry point that computes returns SPG_ERR_NO_DEVICE.
#include <algorithm>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <string>
#include <chrono>
#include <thread>
#include <vector>

#include "spg_ctx.h"
#include "spg_plan.h"

namespace {

thread_local std::string g_err;

struct Bucket {
    std::vector<int32_t> list;
    int max_nv = 0, max_e = 0, max_rec = 0;
};

} // namespace

void spg_set_err(const std::string &s) { g_err = s; }
#define set_err spg_set_err

namespace {

// FP64 pipe peak probe: 8 independent DFMA chains per thread, no memory traffic.
__global__ void __launch_bounds__(256) dfma_probe_kernel(double *sink, int iters, double seed) {
    double a0 = seed + threadIdx.x, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6, a7 = a0 + 7;
    const double m = 1.0000001, c = 1e-9;
    for(int i = 0; i < iters; i++) {
#pragma unroll
        for(int u = 0; u < 8; u++) {
            a0 = fma(a0, m, c); a1 = fma(a1, m, c); a2 = fma(a2, m, c); a3 = fma(a3, m, c);
            a4 = fma(a4, m, c); a5 = fma(a5, m, c); a6 = fma(a6, m, c); a7 = fma(a7, m, c);
        }
    }
    const double r = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
    if(r == 12345.678) sink[0] = r; // never true: keeps the chains alive
}

template <int D>
spg_status launch_general(spg_ctx *ctx, spg::KernelParams &kp);

// NFR tree rounds go through fast_kernel first (spg_fast.cuh); the blankets it refuses (non-POSE edges, several
// removed vertices, a failed guard or pivot) are collected in a device-side list and re-run by blanket_kernel,
// launched right behind it with the count read on the device.
template <int D>
spg_status launch_dim(spg_ctx *ctx, spg::KernelParams &kp) {
    const int nk = kp.max_nv - 1, tiles = nk * (nk + 1) / 2;
    const bool eligible = !ctx->no_fast && kp.algorithm == SPG_ALG_NFR && kp.topology == SPG_TOPO_TREE &&
                          !(kp.flags & SPG_OPT_FORCE_EIGEN) && kp.max_nv >= 3 && tiles <= 256 && kp.retry_list && kp.retry_count;
    if(eligible) {
        spg_status st;
        const int gsel = getenv("SPG_FAST_NOGROUPS") ? 32 : (tiles <= 8 ? 8 : (tiles <= 16 ? 16 : 32)); // sub-warp group width
        if(D == 6) {
            if(tiles <= 32) st = gsel == 8 ? spg_launch_fast_6_g8(ctx, kp) : (gsel == 16 ? spg_launch_fast_6_g16(ctx, kp) : spg_launch_fast_6_g32(ctx, kp));
            else st = tiles <= 128 ? spg_launch_fast_6_c4(ctx, kp) : spg_launch_fast_6_c8(ctx, kp);
        } else {
            if(tiles <= 32) st = gsel == 8 ? spg_launch_fast_3_g8(ctx, kp) : (gsel == 16 ? spg_launch_fast_3_g16(ctx, kp) : spg_launch_fast_3_g32(ctx, kp));
            else st = spg_launch_fast_3_c8(ctx, kp);
        }
        if(st == SPG_OK) {
            spg::KernelParams kr = kp;
            kr.list = kp.retry_list;
            kr.n_list_dev = kp.retry_count;
            return launch_general<D>(ctx, kr);
        }
        if(st != SPG_ERR_UNSUPPORTED) return st;
    }
    kp.n_list_dev = nullptr;
    return launch_general<D>(ctx, kp);
}

template <int D>
spg_status launch_general(spg_ctx *ctx, spg::KernelParams &kp) {
    spg::plan_smem<D>(kp);
    // CTA width by the size of H (N = D * vertices): the register-tiled sweeps cover
    // N <= 12 / 32 / 48 / 96 for 32 / 64 / 128 / 256 threads (SweepGrid in spg_device.cuh)
    const int N = D * kp.max_nv;
    // NFR rounds of POSE edges, 48 < N <= 80: lean variant, two CTAs per SM (falls through when it does not fit twice)
    const bool cliquey = kp.topology == SPG_TOPO_CLIQUEY_SUBGRAPH || kp.topology == SPG_TOPO_CLIQUEY_DENSE; // needs the full third buffer
    if(kp.algorithm == SPG_ALG_NFR && (kp.flags & SPG_OPT_POSE_EDGES_ONLY) && N > 48 && N <= 80 && !cliquey) {
        kp.lean = 1;
        spg::plan_smem<D>(kp);
        const spg_status st = (D == 6) ? spg_launch_6_256l(ctx, kp) : spg_launch_3_256l(ctx, kp);
        if(st != SPG_ERR_UNSUPPORTED) return st;
        kp.lean = 0;
        spg::plan_smem<D>(kp);
    }
    // GLC tree: fewer factor-finishing warps (less scratch) before giving up on shared memory
    while(kp.algorithm == SPG_ALG_GLC && kp.glc_warps > 1 && (size_t) kp.total_doubles * sizeof(double) > ctx->smem_optin) {
        kp.glc_warps--;
        spg::plan_smem<D>(kp);
    }
    // working set beyond shared memory (SE3 > 19, SE2 > 39 vertices): same kernel over a global workspace
    if((size_t) kp.total_doubles * sizeof(double) > ctx->smem_optin)
        return D == 6 ? spg_launch_6_spill(ctx, kp) : spg_launch_3_spill(ctx, kp);
    if(D == 6) {
        if(N <= 12) return spg_launch_6_32(ctx, kp);
        if(N <= 32) return spg_launch_6_64(ctx, kp);
        if(N <= 48) return spg_launch_6_128(ctx, kp);
        if(N <= 80) return spg_launch_6_512(ctx, kp); // 5 x 5 tiles fit the 128 registers of a 512-thread CTA
        return spg_launch_6_256(ctx, kp);
    }
    if(N <= 12) return spg_launch_3_32(ctx, kp);
    if(N <= 32) return spg_launch_3_64(ctx, kp);
    if(N <= 48) return spg_launch_3_128(ctx, kp);
    if(N <= 80) return spg_launch_3_512(ctx, kp);
    return spg_launch_3_256(ctx, kp);
}

// Host-side validation of blankets [b0, b1) of a round: everything the kernels index with (edge offset table,
// edge-local vertex indices, edge sizes, output slice) must lie inside the record / the output slice.
// Returns the index of the first malformed blanket, or -1.
int validate_records(const spg_round_in *in, int b0, int b1, int32_t *hdr3, int hdr_base) {
    const int dim = in->dim;
    for(int b = b0; b < b1; b++) {
        const uint64_t *rec = in->records + in->rec_off[b];
        if(b + 1 < b1) __builtin_prefetch(in->records + in->rec_off[b + 1]);
        const int64_t rw = in->rec_off[b + 1] - in->rec_off[b];
        if(rw < SPG_REC_HEADER_WORDS) return b;
        const int32_t *h = reinterpret_cast<const int32_t *>(rec);
        const int nv = h[0], nrem = h[1], ne = h[2];
        if(hdr3) { // what the bucketing needs, captured while the header is in cache
            int32_t *o = hdr3 + 3 * (size_t) (b - hdr_base);
            o[0] = nv; o[1] = ne; o[2] = h[4];
        }
        if(h[3] != dim || h[4] > rw || h[4] < SPG_REC_HEADER_WORDS || nv < 1 || nrem < 1 || nrem > nv || ne < 0) return b;
        const int64_t words = h[4], fixed = spgr_record_fixed_words(dim, nv, ne);
        if(fixed > words) return b;
        const int32_t *etab = reinterpret_cast<const int32_t *>(rec + spgr_edgetab_off(dim, nv));
        for(int e = 0; e < ne; e++) {
            // the edge headers of a record are a cache line or more apart: fetch a few edges ahead (offsets are checked
            // before use; a wild prefetch address is harmless)
            if(e + 6 < ne) __builtin_prefetch(rec + (etab[e + 6] & 0xffffff));
            const int64_t eo = etab[e];
            if(eo < fixed || eo + 2 > words) return b;
            const int32_t *eh = reinterpret_cast<const int32_t *>(rec + eo);
            const int kind = eh[0], env = eh[1], rows = eh[2];
            if(kind < SPG_EDGE_POSE || kind > SPG_EDGE_MULTI || env < 1 || env > nv || rows < 0) return b;
            if(kind == SPG_EDGE_POSE && (env != 2 || rows != dim)) return b;
            if(kind == SPG_EDGE_GLC && rows > dim * env) return b;
            if(kind == SPG_EDGE_MULTI && rows % dim != 0) return b;
            if(eo + 2 + spgr_pad2(env) > words || eo + spgr_edge_words(dim, kind, env, rows) > words) return b;
            const int32_t *vi = reinterpret_cast<const int32_t *>(rec + eo + 2);
            for(int q = 0; q < env; q++)
                if(vi[q] < 0 || vi[q] >= nv) return b;
            if(kind == SPG_EDGE_MULTI) {
                const int32_t *pr = reinterpret_cast<const int32_t *>(rec + eo + 2 + spgr_pad2(env));
                for(int q = 0; q < 2 * (rows / dim); q++)
                    if(pr[q] < 0 || pr[q] >= env) return b;
            }
        }
        const int64_t need = spgr_out_record_words(dim, in->algorithm, in->opts.topology, in->opts.chord_ratio, nv - nrem);
        if(in->out_off[b + 1] - in->out_off[b] < need) return b;
    }
    return -1;
}

// the same over a large range, spread over host threads (the check of chunk c+1 overlaps the GPU work of chunk c)
int validate_records_mt(const spg_round_in *in, int b0, int b1, int32_t *hdr3, int nranks) {
    const int n = b1 - b0;
    // the ranks of a sharded round share the host: split its cores between them
    unsigned nthr = std::min<unsigned>(std::max(1u, std::thread::hardware_concurrency() / (unsigned) std::max(1, nranks)), 8u);
    if(n < 1024 || nthr <= 1) return validate_records(in, b0, b1, hdr3, b0); // (a sharded rank's pipeline step is a few thousand blankets)
    std::vector<int> bad(nthr, -1);
    std::vector<std::thread> pool;
    const int per = (n + (int) nthr - 1) / (int) nthr;
    for(unsigned t = 0; t < nthr; t++) {
        const int lo = std::min(b1, b0 + (int) t * per), hi = std::min(b1, lo + per);
        if(lo < hi) pool.emplace_back([&bad, in, lo, hi, t, hdr3, b0] { bad[t] = validate_records(in, lo, hi, hdr3, b0); });
    }
    for(auto &th : pool) th.join();
    for(int v : bad)
        if(v >= 0) return v;
    return -1;
}

spg_status check_device(spg_ctx *ctx) {
    if(!ctx) {
        set_err("null context");
        return SPG_ERR_INVALID;
    }
    return SPG_OK;
}

} // namespace

// ---- pieces of the host-buffer round shared by spg_remove_round and spg_remove_round_sharded (spg_comm.cu) ----------

// contiguous split of blankets [b0, b1) into `parts` runs of about equal bytes (records + outputs): parts+1 bounds
void spg_split_by_bytes(const spg_round_in *in, int b0, int b1, int parts, std::vector<int> &cb) {
    cb.assign(parts + 1, b1);
    cb[0] = b0;
    const int64_t base = in->rec_off[b0] + in->out_off[b0];
    const int64_t total = (in->rec_off[b1] + in->out_off[b1] - base) * 8;
    for(int c = 1, b = b0; c < parts; c++) {
        const int64_t goal = total / parts * c;
        while(b < b1 && (in->rec_off[b] + in->out_off[b] - base) * 8 < goal) b++;
        cb[c] = b;
    }
}

// device buffers at the host offsets, offset tables and debug buffers up, retry counters zeroed (stream s_in)
spg_status spg_round_prepare(spg_ctx *ctx, const spg_round_in *in, spg_round_out *out, int nchunks, spg::RoundRun &run) {
    const int nb = in->n_blankets;
    const int64_t rec_words = in->rec_off[nb], out_words = in->out_off[nb];
    if(!ctx->s_in) {
        SPG_CUDA(cudaStreamCreateWithFlags(&ctx->s_in, cudaStreamNonBlocking));
        SPG_CUDA(cudaStreamCreateWithFlags(&ctx->s_out, cudaStreamNonBlocking));
    }
    for(int k = 0; k < spg_ctx::N_SIDE; k++)
        if(!ctx->s_side[k]) {
            SPG_CUDA(cudaStreamCreateWithFlags(&ctx->s_side[k], cudaStreamNonBlocking));
            SPG_CUDA(cudaEventCreateWithFlags(&ctx->ev_side[k], cudaEventDisableTiming));
        }
    while((int) ctx->ev_pool.size() < 2 * nchunks) {
        cudaEvent_t e;
        SPG_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        ctx->ev_pool.push_back(e);
    }
    SPG_CUDA(ctx->d_rec.reserve((size_t) rec_words * 8));
    SPG_CUDA(ctx->d_recoff.reserve((size_t) (nb + 1) * 8));
    SPG_CUDA(ctx->d_outoff.reserve((size_t) (nb + 1) * 8));
    SPG_CUDA(ctx->d_out.reserve((size_t) out_words * 8));
    SPG_CUDA(ctx->d_list.reserve((size_t) nb * 4));
    SPG_CUDA(ctx->d_retry.reserve((size_t) nb * 4));
    const int n_counters = nchunks * 32; // one per bucket launch (NBK <= 32)
    SPG_CUDA(ctx->d_retry_cnt.reserve((size_t) n_counters * 4));
    SPG_CUDA(cudaMemsetAsync(ctx->d_retry_cnt.p, 0, (size_t) n_counters * 4, ctx->s_in));
    run.counter_next = 0;
    run.first = true;
    run.flat.resize(nb);
    SPG_CUDA(cudaMemcpyAsync(ctx->d_recoff.p, in->rec_off, (size_t) (nb + 1) * 8, cudaMemcpyHostToDevice, ctx->s_in));
    SPG_CUDA(cudaMemcpyAsync(ctx->d_outoff.p, in->out_off, (size_t) (nb + 1) * 8, cudaMemcpyHostToDevice, ctx->s_in));
    run.tgt_n = run.wts_n = 0;
    if(out->dbg_target && out->dbg_target_off) {
        run.tgt_n = out->dbg_target_off[nb];
        SPG_CUDA(ctx->d_tgt.reserve((size_t) run.tgt_n * 8 + 8));
        SPG_CUDA(ctx->d_tgtoff.reserve((size_t) (nb + 1) * 8));
        SPG_CUDA(cudaMemcpyAsync(ctx->d_tgtoff.p, out->dbg_target_off, (size_t) (nb + 1) * 8, cudaMemcpyHostToDevice, ctx->s_in));
        SPG_CUDA(cudaMemsetAsync(ctx->d_tgt.p, 0, (size_t) run.tgt_n * 8 + 8, ctx->s_in));
    }
    if(out->dbg_weights && out->dbg_weights_off) {
        run.wts_n = out->dbg_weights_off[nb];
        SPG_CUDA(ctx->d_wts.reserve((size_t) run.wts_n * 8 + 8));
        SPG_CUDA(ctx->d_wtsoff.reserve((size_t) (nb + 1) * 8));
        SPG_CUDA(cudaMemcpyAsync(ctx->d_wtsoff.p, out->dbg_weights_off, (size_t) (nb + 1) * 8, cudaMemcpyHostToDevice, ctx->s_in));
        if(in->opts.flags & SPG_OPT_DBG_WEIGHTS_IN)
            SPG_CUDA(cudaMemcpyAsync(ctx->d_wts.p, out->dbg_weights, (size_t) run.wts_n * 8, cudaMemcpyHostToDevice, ctx->s_in));
        else
            SPG_CUDA(cudaMemsetAsync(ctx->d_wts.p, 0, (size_t) run.wts_n * 8 + 8, ctx->s_in));
    }
    return SPG_OK;
}

namespace {
// SPG_HOST_PROF=1: where the host time of the round calls goes (printed at exit)
struct CapiProf {
    double prepare = 0, fill = 0, validate = 0, bucket = 0, enqueue = 0, finish = 0, drain = 0;
    long long rounds = 0, chunks = 0;
    bool on = getenv("SPG_HOST_PROF") != nullptr;
    ~CapiProf() {
        if(on && rounds)
            fprintf(stderr, "[spg capi] %lld round calls, %lld chunks: prepare %.3f s, fill callback %.3f s, validate %.3f s, bucket %.3f s, "
                            "copies + launches enqueued %.3f s, drain callback incl. its waits %.3f s, final wait %.3f s\n", rounds, chunks, prepare, fill, validate, bucket, enqueue,
                    drain, finish);
    }
} g_cprof;
inline double now_s() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }
} // namespace

// blankets [b0, b1) of the round: validate, bucket by size, H2D on s_in (event 2c), one fused kernel per bucket on
// the context stream (event 2c+1 behind the last one)
spg_status spg_round_enqueue_chunk(spg_ctx *ctx, const spg_round_in *in, spg::RoundRun &run, int b0, int b1, int c) {
    static const int bounds6[] = {3, 4, 5, 6, 7, 8, 10, 12, 14, 16, 20, 24, 32, 48, 64, 128, 1 << 30};
    constexpr int NBK = sizeof(bounds6) / sizeof(int);
    const int dim = in->dim;
    std::vector<int32_t> hdr3; // (n_vert, n_edges, rec_words) of every blanket of the chunk
    double tp = now_s();
    g_cprof.chunks++;
    // ---- validate the chunk's records before anything of it is launched (runs while the GPU works on c-1)
    {
        hdr3.resize(3 * (size_t) (b1 - b0));
        const int bad = validate_records_mt(in, b0, b1, hdr3.data(), ctx->nranks);
        if(bad >= 0) {
            cudaDeviceSynchronize();
            set_err("malformed blanket record " + std::to_string(bad) +
                    " (header, edge table, vertex index or output slice out of bounds)");
            return SPG_ERR_INVALID;
        }
    }
    g_cprof.validate += now_s() - tp; tp = now_s();
    // ---- bucket this chunk by blanket size -----------------------------------------------------
    std::vector<Bucket> buckets(NBK);
    for(int b = b0; b < b1; b++) {
        const int32_t *h = hdr3.data() + 3 * (size_t) (b - b0);
        int bi = 0;
        while(h[0] > bounds6[bi]) bi++;
        Bucket &B = buckets[bi];
        B.list.push_back(b);
        B.max_nv = std::max(B.max_nv, (int) h[0]);
        B.max_e = std::max(B.max_e, (int) h[1]);
        B.max_rec = std::max(B.max_rec, (int) h[2]);
    }
    size_t pos = (size_t) b0;
    for(auto &B : buckets) {
        std::copy(B.list.begin(), B.list.end(), run.flat.begin() + pos);
        pos += B.list.size();
    }
    g_cprof.bucket += now_s() - tp; tp = now_s();
    // ---- H2D of the chunk -----------------------------------------------------------------------
    const int64_t r0 = in->rec_off[b0], r1 = in->rec_off[b1];
    SPG_CUDA(cudaMemcpyAsync(reinterpret_cast<uint64_t *>(ctx->d_rec.p) + r0, in->records + r0, (size_t) (r1 - r0) * 8,
                             cudaMemcpyHostToDevice, ctx->s_in));
    SPG_CUDA(cudaMemcpyAsync(reinterpret_cast<int32_t *>(ctx->d_list.p) + b0, run.flat.data() + b0, (size_t) (b1 - b0) * 4,
                             cudaMemcpyHostToDevice, ctx->s_in));
    SPG_CUDA(cudaEventRecord(ctx->ev_pool[2 * c], ctx->s_in));
    SPG_CUDA(cudaStreamWaitEvent(ctx->stream, ctx->ev_pool[2 * c], 0));
    if(run.first) {
        SPG_CUDA(cudaEventRecord(ctx->ev0, ctx->stream));
        run.first = false;
    }
    // ---- kernels ----------------------------------------------------------------------------------
    // NFR tree rounds of on-chip blankets use no per-context workspace: their buckets go round-robin to the side
    // streams and run side by side (a graph-level round holds blankets of many sizes, and a bucket of a few hundred
    // blankets fills a fraction of the SMs); everything else runs bucket after bucket on the context stream
    int n_buckets = 0;
    for(auto &B : buckets) n_buckets += !B.list.empty();
    static const bool no_side = getenv("SPG_NO_SIDE_STREAMS") != nullptr;
    const bool side = !no_side && n_buckets > 1 && in->algorithm == SPG_ALG_NFR && in->opts.topology == SPG_TOPO_TREE &&
                      !ctx->profiling && ctx->s_side[0];
    cudaStream_t const main_stream = ctx->stream;
    bool used_side[spg_ctx::N_SIDE] = {};
    int next_side = 0;
    size_t list_pos = (size_t) b0;
    for(auto &B : buckets) {
        if(B.list.empty()) continue;
        const bool on_side = side && B.max_nv <= 16; // (far below the spill limit: no global workspace)
        if(on_side) {
            const int k = next_side++ % spg_ctx::N_SIDE;
            if(!used_side[k]) {
                // behind the copy-in of this chunk and behind everything already queued on the context stream
                SPG_CUDA(cudaStreamWaitEvent(ctx->s_side[k], ctx->ev_pool[2 * c], 0));
                SPG_CUDA(cudaEventRecord(ctx->ev_side[k], main_stream));
                SPG_CUDA(cudaStreamWaitEvent(ctx->s_side[k], ctx->ev_side[k], 0));
                used_side[k] = true;
            }
            ctx->stream = ctx->s_side[k];
        }
        spg::KernelParams kp{};
        kp.algorithm = in->algorithm;
        kp.topology = in->opts.topology;
        kp.chord_ratio = in->opts.chord_ratio;
        kp.flags = in->opts.flags;
        kp.n_list = (int32_t) B.list.size();
        kp.list = reinterpret_cast<const int32_t *>(ctx->d_list.p) + list_pos;
        kp.retry_list = reinterpret_cast<int32_t *>(ctx->d_retry.p) + list_pos;
        kp.retry_count = reinterpret_cast<int32_t *>(ctx->d_retry_cnt.p) + run.counter_next++;
        list_pos += B.list.size();
        kp.rec_off = reinterpret_cast<const int64_t *>(ctx->d_recoff.p);
        kp.records = reinterpret_cast<const uint64_t *>(ctx->d_rec.p);
        kp.out_off = reinterpret_cast<const int64_t *>(ctx->d_outoff.p);
        kp.out = reinterpret_cast<uint64_t *>(ctx->d_out.p);
        kp.dbg_target = run.tgt_n ? reinterpret_cast<double *>(ctx->d_tgt.p) : nullptr;
        kp.dbg_target_off = run.tgt_n ? reinterpret_cast<const int64_t *>(ctx->d_tgtoff.p) : nullptr;
        kp.dbg_weights = run.wts_n ? reinterpret_cast<double *>(ctx->d_wts.p) : nullptr;
        kp.dbg_weights_off = run.wts_n ? reinterpret_cast<const int64_t *>(ctx->d_wtsoff.p) : nullptr;
        kp.max_nv = B.max_nv;
        kp.max_e = B.max_e;
        kp.max_rec_words = (B.max_rec + 1) & ~1;
        spg_status st = (dim == 6) ? launch_dim<6>(ctx, kp) : launch_dim<3>(ctx, kp);
        ctx->stream = main_stream;
        if(st != SPG_OK) {
            cudaDeviceSynchronize();
            return st;
        }
    }
    for(int k = 0; k < spg_ctx::N_SIDE; k++) // join: the chunk is done when every side stream is
        if(used_side[k]) {
            SPG_CUDA(cudaEventRecord(ctx->ev_side[k], ctx->s_side[k]));
            SPG_CUDA(cudaStreamWaitEvent(main_stream, ctx->ev_side[k], 0));
        }
    SPG_CUDA(cudaEventRecord(ctx->ev_pool[2 * c + 1], ctx->stream));
    g_cprof.enqueue += now_s() - tp;
    return SPG_OK;
}

// debug buffers back, all three streams drained, kernel time of the call recorded
spg_status spg_round_finish(spg_ctx *ctx, spg_round_out *out, spg::RoundRun &run) {
    ctx->retry_used = run.counter_next;
    SPG_CUDA(cudaEventRecord(ctx->ev1, ctx->stream));
    if(run.tgt_n) SPG_CUDA(cudaMemcpyAsync(out->dbg_target, ctx->d_tgt.p, (size_t) run.tgt_n * 8, cudaMemcpyDeviceToHost, ctx->s_out));
    if(run.wts_n) SPG_CUDA(cudaMemcpyAsync(out->dbg_weights, ctx->d_wts.p, (size_t) run.wts_n * 8, cudaMemcpyDeviceToHost, ctx->s_out));
    SPG_CUDA(cudaStreamSynchronize(ctx->s_in));
    SPG_CUDA(cudaStreamSynchronize(ctx->stream));
    SPG_CUDA(cudaStreamSynchronize(ctx->s_out));
    float ms = 0;
    if(!run.first) {
        SPG_CUDA(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
        ctx->last_ms = ms; // first kernel to last kernel of the call (waits for the chunked copies included)
    }
    return SPG_OK;
}

uint64_t *spg_ctx_pinned(spg_ctx *ctx, int slot, size_t words) {
    if(!ctx || slot < 0 || slot > 1) return nullptr;
    if(words <= ctx->h_pinned_words[slot]) return static_cast<uint64_t *>(ctx->h_pinned[slot]);
    cudaSetDevice(ctx->device);
    if(ctx->h_pinned[slot]) cudaFreeHost(ctx->h_pinned[slot]);
    ctx->h_pinned[slot] = nullptr;
    ctx->h_pinned_words[slot] = 0;
    // page-locking costs ~0.3 ms per MB: grow by doubling from 8 MB so that a removal re-pins at most a couple of times
    const size_t want = std::max<size_t>(2 * words, (size_t) 1 << 20);
    void *q = nullptr;
    if(cudaHostAlloc(&q, want * 8, cudaHostAllocDefault) != cudaSuccess) {
        (void) cudaGetLastError();
        return nullptr;
    }
    ctx->h_pinned[slot] = q;
    ctx->h_pinned_words[slot] = want;
    return static_cast<uint64_t *>(q);
}

extern "C" {

const char *spg_version(void) { return "sparsifyposegraph_b200 0.1 (sm_100a)"; }
const char *spg_last_error(void) { return g_err.c_str(); }

spg_status spg_create(spg_ctx **out, const spg_config *cfg) {
    if(!out) return SPG_ERR_INVALID;
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if(e != cudaSuccess || count == 0) {
        set_err("no CUDA device: the node-removal path has no CPU fallback");
        return SPG_ERR_NO_DEVICE;
    }
    int dev = cfg ? cfg->device : 0;
    if(dev < 0 || dev >= count) {
        set_err("bad device ordinal");
        return SPG_ERR_INVALID;
    }
    cudaDeviceProp prop;
    SPG_CUDA(cudaGetDeviceProperties(&prop, dev));
    if(prop.major < 10) {
        set_err(std::string("device is sm_") + std::to_string(prop.major) + std::to_string(prop.minor) +
                ", this library is built for sm_100a only");
        return SPG_ERR_NO_DEVICE;
    }
    SPG_CUDA(cudaSetDevice(dev));
    spg_ctx *ctx = new spg_ctx;
    ctx->device = dev;
    ctx->sm_count = prop.multiProcessorCount;
    ctx->smem_optin = prop.sharedMemPerBlockOptin;
    if(const char *e = getenv("SPG_NO_FAST")) ctx->no_fast = atoi(e) != 0;
    if(const char *e = getenv("SPG_CHUNK_BYTES")) ctx->chunk_bytes = std::max<long long>(4096, atoll(e)); // tests: force many chunks
    // SPG_OPT_DENSE_MAX_DIMS (tests: the optimiser's block-sparse path on small graphs) is read by every
    // spg_graph_optimize call instead (spg_eval.cu, dense_fits), so it can change after the context exists
    SPG_CUDA(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
    SPG_CUDA(cudaEventCreate(&ctx->ev0));
    SPG_CUDA(cudaEventCreate(&ctx->ev1));
    if(cfg && cfg->max_record_words > 0) SPG_CUDA(ctx->d_rec.reserve((size_t) cfg->max_record_words * 8));
    if(cfg && cfg->max_out_words > 0) SPG_CUDA(ctx->d_out.reserve((size_t) cfg->max_out_words * 8));
    *out = ctx;
    return SPG_OK;
}

void spg_destroy(spg_ctx *ctx) {
    if(!ctx) return;
    cudaSetDevice(ctx->device);
    spg_comm_release(ctx);
    for(DevBuf *b : {&ctx->d_rec, &ctx->d_recoff, &ctx->d_outoff, &ctx->d_out, &ctx->d_list, &ctx->d_tgt,
                     &ctx->d_tgtoff, &ctx->d_wts, &ctx->d_wtsoff, &ctx->d_ws, &ctx->d_gws, &ctx->d_prof, &ctx->d_retry, &ctx->d_retry_cnt})
        b->release();
    for(void *&hp : ctx->h_pinned) {
        if(hp) cudaFreeHost(hp);
        hp = nullptr;
    }
    if(ctx->ev0) cudaEventDestroy(ctx->ev0);
    if(ctx->ev1) cudaEventDestroy(ctx->ev1);
    for(cudaEvent_t e : ctx->ev_pool) cudaEventDestroy(e);
    for(int k = 0; k < spg_ctx::N_SIDE; k++) {
        if(ctx->s_side[k]) cudaStreamDestroy(ctx->s_side[k]);
        if(ctx->ev_side[k]) cudaEventDestroy(ctx->ev_side[k]);
    }
    if(ctx->s_in) cudaStreamDestroy(ctx->s_in);
    if(ctx->s_out) cudaStreamDestroy(ctx->s_out);
    if(ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

spg_status spg_reserve_staging(spg_ctx *ctx, int64_t record_words, int64_t out_words) {
    if(check_device(ctx) != SPG_OK || record_words < 0 || out_words < 0) return SPG_ERR_INVALID;
    if(record_words > 0 && !spg_ctx_pinned(ctx, 0, (size_t) record_words)) {
        set_err("cannot page-lock the record staging buffer");
        return SPG_ERR_CUDA;
    }
    if(out_words > 0 && !spg_ctx_pinned(ctx, 1, (size_t) out_words)) {
        set_err("cannot page-lock the output staging buffer");
        return SPG_ERR_CUDA;
    }
    return SPG_OK;
}
int64_t spg_launch_count(const spg_ctx *ctx) { return ctx ? ctx->launches : 0; }
double spg_last_kernel_ms(const spg_ctx *ctx) { return ctx ? ctx->last_ms : 0.0; }
void *spg_stream(spg_ctx *ctx) { return ctx ? (void *) ctx->stream : nullptr; }

int64_t spg_pose_words(int32_t dim) { return spgr_pose_words(dim); }
int64_t spg_record_words(int32_t dim, int32_t n_vert, int32_t n_edges, const int32_t *edge_kind,
                         const int32_t *edge_nv, const int32_t *edge_rows) {
    int64_t w = spgr_record_fixed_words(dim, n_vert, n_edges);
    for(int e = 0; e < n_edges; e++) w += spgr_edge_words(dim, edge_kind[e], edge_nv[e], edge_rows[e]);
    return (w + 1) & ~(int64_t) 1;
}
int64_t spg_out_record_words(int32_t dim, int32_t algorithm, const spg_sparsity_options *o, int32_t n_kept) {
    return spgr_out_record_words(dim, algorithm, o->topology, o->chord_ratio, n_kept);
}
int32_t spg_out_edge_count(int32_t algorithm, const spg_sparsity_options *o, int32_t n_kept) {
    return spgr_out_edge_count(algorithm, o->topology, o->chord_ratio, n_kept);
}
int64_t spg_out_slot_words(int32_t dim, int32_t algorithm, const spg_sparsity_options *o, int32_t n_kept) {
    return spgr_out_slot_words(dim, algorithm, o->topology, n_kept);
}

spg_status spg_fp64_peak_probe(spg_ctx *ctx, int32_t repeats, double *tflops) {
    if(check_device(ctx) != SPG_OK || !tflops) return SPG_ERR_INVALID;
    SPG_CUDA(cudaSetDevice(ctx->device));
    SPG_CUDA(ctx->d_list.reserve(64));
    const int iters = 4096, blocks = ctx->sm_count * 8, threads = 256;
    double best = 0;
    for(int r = 0; r < repeats + 1; r++) {
        SPG_CUDA(cudaEventRecord(ctx->ev0, ctx->stream));
        dfma_probe_kernel<<<blocks, threads, 0, ctx->stream>>>(reinterpret_cast<double *>(ctx->d_list.p), iters, 1.0 + r);
        SPG_CUDA(cudaGetLastError());
        SPG_CUDA(cudaEventRecord(ctx->ev1, ctx->stream));
        SPG_CUDA(cudaStreamSynchronize(ctx->stream));
        ctx->launches++;
        float ms = 0;
        SPG_CUDA(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
        const double flops = 2.0 * 64.0 * iters * (double) blocks * threads;
        if(r > 0) best = std::max(best, flops / (ms * 1e-3) / 1e12);
    }
    *tflops = best;
    return SPG_OK;
}

// Developer aid: per-stage cycle accumulators (thread 0 of every CTA, clock64): [0,16) blanket_kernel, [16,32)
// fast_kernel. enable != 0 zeroes and enables them; cycles (32 values) may be NULL. Not part of the product path.
spg_status spg_stage_profile(spg_ctx *ctx, int32_t enable, uint64_t *cycles) {
    if(check_device(ctx) != SPG_OK) return SPG_ERR_INVALID;
    SPG_CUDA(cudaSetDevice(ctx->device));
    SPG_CUDA(ctx->d_prof.reserve(32 * 8));
    SPG_CUDA(cudaStreamSynchronize(ctx->stream));
    if(cycles) SPG_CUDA(cudaMemcpy(cycles, ctx->d_prof.p, 32 * 8, cudaMemcpyDeviceToHost));
    if(enable) SPG_CUDA(cudaMemset(ctx->d_prof.p, 0, 32 * 8));
    ctx->profiling = enable != 0;
    return SPG_OK;
}

// Diagnostics: blankets of the last spg_remove_round* call that fast_kernel handed over to blanket_kernel
// (synchronises the context's stream).
int64_t spg_last_retry_count(spg_ctx *ctx) {
    if(!ctx || ctx->retry_used <= 0 || !ctx->d_retry_cnt.p) return 0;
    cudaSetDevice(ctx->device);
    if(cudaStreamSynchronize(ctx->stream) != cudaSuccess) return -1;
    std::vector<int32_t> h((size_t) ctx->retry_used);
    if(cudaMemcpy(h.data(), ctx->d_retry_cnt.p, h.size() * 4, cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
    int64_t t = 0;
    for(int32_t v : h) t += v;
    return t;
}

spg_status spg_sync(spg_ctx *ctx) {
    if(check_device(ctx) != SPG_OK) return SPG_ERR_INVALID;
    SPG_CUDA(cudaStreamSynchronize(ctx->stream));
    if(ctx->s_comm) SPG_CUDA(cudaStreamSynchronize(ctx->s_comm));
    float ms = 0;
    if(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1) == cudaSuccess) ctx->last_ms = ms;
    else (void) cudaGetLastError();
    return SPG_OK;
}

spg_status spg_remove_round_device(spg_ctx *ctx, const spg_round_in *in, spg_round_out *out, int32_t max_n_vert,
                                   int32_t max_n_edges, int32_t max_rec_words) {
    if(check_device(ctx) != SPG_OK) return SPG_ERR_INVALID;
    if(!in || !out || (in->dim != 3 && in->dim != 6)) {
        set_err("bad round descriptor");
        return SPG_ERR_INVALID;
    }
    SPG_CUDA(cudaSetDevice(ctx->device));
    spg::KernelParams kp{};
    kp.algorithm = in->algorithm;
    kp.topology = in->opts.topology;
    kp.chord_ratio = in->opts.chord_ratio;
    kp.flags = in->opts.flags;
    kp.n_list = in->n_blankets;
    kp.list = nullptr;
    kp.rec_off = in->rec_off;
    kp.records = in->records;
    kp.out_off = in->out_off;
    kp.out = out->out;
    kp.dbg_target = out->dbg_target;
    kp.dbg_target_off = out->dbg_target_off;
    kp.dbg_weights = out->dbg_weights;
    kp.dbg_weights_off = out->dbg_weights_off;
    kp.max_nv = max_n_vert;
    kp.max_e = max_n_edges;
    // record size bound: from the caller (rounds with GLC / MULTI edges), else the all-POSE bound for this (nv, ne)
    kp.max_rec_words = max_rec_words > 0 ? ((max_rec_words + 1) & ~1)
                                         : (int32_t) ((spgr_record_fixed_words(in->dim, max_n_vert, max_n_edges) +
                                   (int64_t) max_n_edges * spgr_edge_words(in->dim, SPG_EDGE_POSE, 2, in->dim) + 1) & ~1LL);
    SPG_CUDA(ctx->d_retry.reserve((size_t) std::max(1, in->n_blankets) * 4));
    SPG_CUDA(ctx->d_retry_cnt.reserve(64));
    SPG_CUDA(cudaMemsetAsync(ctx->d_retry_cnt.p, 0, 4, ctx->stream));
    kp.retry_list = reinterpret_cast<int32_t *>(ctx->d_retry.p);
    kp.retry_count = reinterpret_cast<int32_t *>(ctx->d_retry_cnt.p);
    ctx->retry_used = 1;
    SPG_CUDA(cudaEventRecord(ctx->ev0, ctx->stream));
    spg_status st = (in->dim == 6) ? launch_dim<6>(ctx, kp) : launch_dim<3>(ctx, kp);
    if(st != SPG_OK) return st;
    SPG_CUDA(cudaEventRecord(ctx->ev1, ctx->stream));
    return SPG_OK;
}

spg_status spg_remove_round(spg_ctx *ctx, const spg_round_in *in, spg_round_out *out) {
    return spg_remove_round_streamed(ctx, in, out, nullptr, nullptr);
}

spg_status spg_remove_round_streamed(spg_ctx *ctx, const spg_round_in *in, spg_round_out *out, spg_fill_fn fill, void *user) {
    return spg_remove_round_pipelined(ctx, in, out, fill, nullptr, user);
}

spg_status spg_remove_round_pipelined(spg_ctx *ctx, const spg_round_in *in, spg_round_out *out, spg_fill_fn fill, spg_drain_fn drain,
                                      void *user) {
    if(check_device(ctx) != SPG_OK) return SPG_ERR_INVALID;
    if(!in || !out || !out->out || (in->dim != 3 && in->dim != 6) || in->n_blankets < 0) {
        set_err("bad round descriptor");
        return SPG_ERR_INVALID;
    }
    const int nb = in->n_blankets;
    if(nb == 0) return SPG_OK;
    if(!in->rec_off || !in->out_off || !in->records) {
        set_err("bad round descriptor");
        return SPG_ERR_INVALID;
    }
    SPG_CUDA(cudaSetDevice(ctx->device));
    const int64_t rec_words = in->rec_off[nb];
    const int64_t out_words = in->out_off[nb];

    // ---- chunks: contiguous runs of blankets, so that the H2D copy of chunk c+1, the kernels of chunk c and the
    // D2H copy of chunk c-1 overlap (three streams, events in between). Every chunk owns its own slice of the
    // device buffers (same offsets as on the host), so nothing is double-buffered. Small rounds: one chunk.
    const bool dbg = (out->dbg_target && out->dbg_target_off) || (out->dbg_weights && out->dbg_weights_off);
    const int64_t total_bytes = (rec_words + out_words) * 8;
    int nchunks = (int) std::min<int64_t>(32, total_bytes / std::max<int64_t>(ctx->chunk_bytes, 4096));
    if(nchunks < 1 || dbg) nchunks = 1;
    std::vector<int> cb;
    spg_split_by_bytes(in, 0, nb, nchunks, cb);

    spg::RoundRun run;
    double tp = now_s();
    g_cprof.rounds++;
    spg_status st = spg_round_prepare(ctx, in, out, nchunks, run);
    if(st != SPG_OK) return st;
    if(drain) // one more event per chunk: its output records have arrived on the host
        while((int) ctx->ev_pool.size() < 3 * nchunks) {
            cudaEvent_t e;
            SPG_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
            ctx->ev_pool.push_back(e);
        }
    g_cprof.prepare += now_s() - tp;
    // chunks whose records are on their way back, in order; drained as their copies complete: between two fills when a
    // copy happens to be done, after the last fill one by one (the host would only wait for the device otherwise)
    std::vector<int> inflight;
    size_t drained = 0;
    auto drain_ready = [&](bool wait) -> spg_status {
        while(drain && drained < inflight.size()) {
            const int c = inflight[drained];
            cudaEvent_t ev = ctx->ev_pool[2 * nchunks + c];
            if(wait) SPG_CUDA(cudaEventSynchronize(ev));
            else {
                const cudaError_t q = cudaEventQuery(ev);
                if(q == cudaErrorNotReady) {
                    (void) cudaGetLastError(); // "not ready" is recorded as the thread's last error: clear it
                    return SPG_OK;
                }
                SPG_CUDA(q);
            }
            const double td = now_s();
            const int rc = drain(user, cb[c], cb[c + 1]);
            g_cprof.drain += now_s() - td;
            if(rc != 0) {
                cudaDeviceSynchronize();
                set_err("the record consumer of spg_remove_round_pipelined failed on blankets [" + std::to_string(cb[c]) + ", " +
                        std::to_string(cb[c + 1]) + ")");
                return SPG_ERR_INVALID;
            }
            drained++;
        }
        return SPG_OK;
    };
    for(int c = 0; c < nchunks; c++) {
        const int b0 = cb[c], b1 = cb[c + 1];
        if(b1 <= b0) continue;
        // streamed rounds: the caller writes the records of this chunk now, while the GPU works on the previous ones
        tp = now_s();
        const int frc = fill ? fill(user, b0, b1) : 0;
        g_cprof.fill += now_s() - tp;
        if(frc != 0) {
            cudaDeviceSynchronize();
            set_err("the record producer of spg_remove_round_streamed failed on blankets [" + std::to_string(b0) + ", " +
                    std::to_string(b1) + ")");
            return SPG_ERR_INVALID;
        }
        st = spg_round_enqueue_chunk(ctx, in, run, b0, b1, c);
        if(st != SPG_OK) return st;
        // ---- D2H of the chunk -----------------------------------------------------------------------
        SPG_CUDA(cudaStreamWaitEvent(ctx->s_out, ctx->ev_pool[2 * c + 1], 0));
        const int64_t o0 = in->out_off[b0], o1 = in->out_off[b1];
        SPG_CUDA(cudaMemcpyAsync(out->out + o0, reinterpret_cast<uint64_t *>(ctx->d_out.p) + o0, (size_t) (o1 - o0) * 8,
                                 cudaMemcpyDeviceToHost, ctx->s_out));
        if(drain) {
            SPG_CUDA(cudaEventRecord(ctx->ev_pool[2 * nchunks + c], ctx->s_out));
            inflight.push_back(c);
            st = drain_ready(false);
            if(st != SPG_OK) return st;
        }
    }
    tp = now_s();
    st = drain_ready(true);
    if(st != SPG_OK) return st;
    const double tdr = now_s() - tp;
    st = spg_round_finish(ctx, out, run);
    g_cprof.finish += now_s() - tp - tdr;
    return st;
}

} // extern "C"
