/*
 * spg_capi.h — C ABI of the B200-native node-removal path (libspg_b200.so).
 *
 * This is the drop-in boundary for the hot path that the reference enters through
 *   GraphWrapperG2O::marginalizeNoOptimize()  (reference src/graph_wrapper_g2o.cpp:398-453)
 *     -> VertexRemover::remove(removeList)    (reference src/vertex_remover.cpp:83-140).
 *
 * Two levels are exported:
 *   1. Blanket level  (spg_remove_round*)  — one wavefront round of non-interfering Markov
 *      blankets, packed into fp64/int32 records, processed by the sm_100a kernels. This is what a
 *      VertexRemover adapter inside the reference would call once per round.
 *   2. Graph level    (spg_graph_*)        — a g2o-free pose-graph container with the reference's
 *      removal semantics (VertexRemover / TopologyProvider / SparsityOptions / decimation),
 *      implemented in C++ on top of level 1. It replaces GraphWrapper::marginalize for callers
 *      that do not bring g2o.
 *
 * Plain pointers and sizes only; no C++ / torch types. All matrices are fp64.
 * Every function returns spg_status; per-blanket numerical conditions are reported in the
 * blanket's output record (never by assert()/exit() as the reference does,
 * src/optimizer.cpp:75-77, src/topology_provider_glc.cpp:85-89).
 */
#ifndef SPG_CAPI_H_
#define SPG_CAPI_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ------------------------------------------------------------------------------------------ */
/* Enumerations                                                                               */
/* ------------------------------------------------------------------------------------------ */

typedef enum {
    SPG_OK = 0,
    SPG_ERR_INVALID = 1,      /* bad argument / malformed record                          */
    SPG_ERR_CUDA = 2,         /* CUDA runtime error (message via spg_last_error)          */
    SPG_ERR_NO_DEVICE = 3,    /* no sm_100 device: the product path has NO CPU fallback   */
    SPG_ERR_UNSUPPORTED = 4,  /* option combination the reference asserts against         */
    SPG_ERR_IO = 5,
    SPG_ERR_BLANKET_FAILED = 6, /* graph level: at least one blanket came back with a status != SPG_BLANKET_OK
                                  (the reference asserts / exits there). Its vertex and edges were left in the
                                  graph untouched; every other removal was applied. spg_marginalize_stats
                                  names the first failing list index and its blanket status.             */
    SPG_ERR_COMM = 7           /* NCCL missing or a collective failed (message via spg_last_error)        */
} spg_status;

/* reference src/sparsity_options.h:12-14 (same numeric values) */
typedef enum {
    SPG_TOPO_TREE = 0,
    SPG_TOPO_SUBGRAPH = 1,
    SPG_TOPO_CLIQUEY_SUBGRAPH = 2,
    SPG_TOPO_DENSE = 3,
    SPG_TOPO_CLIQUEY_DENSE = 4
} spg_topology;

/* reference src/sparsity_options.h:16-18 */
typedef enum { SPG_LIN_LOCAL = 0, SPG_LIN_GLOBAL = 1 } spg_lin_point;

/* which TopologyProvider family is registered, reference src/graph_wrapper_g2o.cpp:431-439 */
typedef enum { SPG_ALG_NFR = 0, SPG_ALG_GLC = 1 } spg_algorithm;

/* reference src/sparsity_options.h:11-30; defaults: Tree, 1.0, Local, true */
typedef struct {
    int32_t topology;             /* spg_topology  */
    int32_t lin_point;            /* spg_lin_point */
    double  chord_ratio;
    int32_t include_intra_clique;
    int32_t flags;                /* library extension, 0 = default. SPG_OPT_FORCE_EIGEN: always run the
                                     eigen-decomposition NFR path (disable the gauge shortcut, DESIGN.md) */
} spg_sparsity_options;
#define SPG_OPT_FORCE_EIGEN 1
/* The caller guarantees that every blanket edge of the round is a POSE edge (no GLC / MULTI factors): NFR rounds
 * of mid-sized blankets then run a leaner kernel, two blankets per SM. A record that breaks the promise is
 * answered with SPG_BLANKET_UNSUPPORTED, never with wrong numbers. VertexRemover sets it per round. */
#define SPG_OPT_POSE_EDGES_ONLY 2

/* Test hook: spg_round_out.dbg_weights is an INPUT — the Chow-Liu mutual-information weights of every blanket
 * (pairs in (i<j) lexicographic order) are taken from it instead of being computed. Lets a test feed exactly
 * equal weights and compare the spanning tree with std::priority_queue's pop order (pseudo_chow_liu.h:49-53). */
#define SPG_OPT_DBG_WEIGHTS_IN 4

/* edge kinds inside a blanket record */
typedef enum {
    SPG_EDGE_POSE = 0,   /* EdgeSE2ISAM (src/se2_compatibility.h:21-52) or EdgeSE3ISAM == g2o::EdgeSE3 */
    SPG_EDGE_GLC = 1,    /* GLCEdge (src/glc_edge.h:15-70), error W * r(x (-) meas), Omega = I    */
    SPG_EDGE_MULTI = 2   /* MultiEdgeCorrelated<E> (src/multi_edge_correlated.h:16-127)           */
} spg_edge_kind;

/* per-blanket status word in the output record */
typedef enum {
    SPG_BLANKET_OK = 0,
    SPG_BLANKET_NOT_PD_MARGINAL = 1,  /* LLT(Lambda_mm) failed, vertex_remover.cpp:444            */
    SPG_BLANKET_NOT_PD_CHOWLIU = 2,   /* LLT(Lambda_t + I) failed, pseudo_chow_liu.cpp:189        */
    SPG_BLANKET_EIG_NOCONV = 3,       /* eigen-solver did not converge                            */
    SPG_BLANKET_NOT_PD_CLOSED = 4,    /* LLT(J Sigma J^T) failed, logdet_function.cpp:273         */
    SPG_BLANKET_TOO_LARGE = 5,        /* iterative-fit workspace of the blanket exceeds its budget */
    SPG_BLANKET_LINESEARCH_FAIL = 6,  /* pqn/line_search.cpp:24-26 returned -1 (ignored by ref.)  */
    SPG_BLANKET_KLD_INF = 7,          /* optimizer.cpp:75-77 (reference calls exit(0))            */
    SPG_BLANKET_UNSUPPORTED = 8,      /* edge kind / option not handled on device                 */
    SPG_BLANKET_NOT_PD_JOINT = 9      /* LLT in PseudoChowLiu::marginal failed (GLC tree)         */
} spg_blanket_status;

/* ------------------------------------------------------------------------------------------ */
/* Packed blanket records (one round).  Unit: 8-byte words.                                   */
/* ------------------------------------------------------------------------------------------ */
/*
 * INPUT record of one blanket (contiguous, 16-byte aligned start; all offsets in words):
 *   w0  : int32 n_vert      | int32 n_removed      vertices: removed first, then kept in
 *   w1  : int32 n_edges     | int32 dim (3|6)       ascending original id (vertex_remover.cpp:349-356)
 *   w2  : int32 rec_words   | int32 flags
 *   w3  : int32 tag         | int32 reserved        tag = caller cookie (index in the removal list)
 *   then int32 vert_id[n_vert]        (padded to a whole word)   original ids
 *   then double pose[n_vert][P]       P = 3 (SE2: x y theta) or 7 (SE3: tx ty tz qx qy qz qw)
 *   then int32 edge_off[n_edges]      (padded)   word offset of each edge from the record start
 *   then edges, each:
 *        e0 : int32 kind | int32 nv                 nv = #vertices of the edge
 *        e1 : int32 rows | int32 reserved           rows = error dimension (d for POSE)
 *        int32 vidx[nv] (padded)                    local vertex indices into this blanket
 *        POSE : double meas[P], double info[d*d]    (column-major, full)
 *        GLC  : double meas[d*nv], double W[rows][d*nv]   (row-major: one constraint per row)
 *   Edge order inside the record is the summation order of H = sum J^T Omega J.
 *
 * OUTPUT record of one blanket:
 *   w0 : int32 status | int32 n_new_edges
 *   w1 : int32 newton_iters | int32 flags   (bit 0: a line search of the iterative fit failed, bit 1: KLD infinite;
 *                                           diagnostics: bit 4: gauge shortcut refused, eigen path taken,
 *                                           bit 5: anchored block not positive definite, bit 6: |diag| >= 1e8,
 *                                           bit 7: two Chow-Liu weights exactly equal, priority_queue order replayed)
 *   w2 : double kld        (value of the projected KLD at the solution, NFR only)
 *   w3 : double reserved
 *   then n_new_edges slots, slot size fixed per (algorithm, dim, topology):
 *     NFR slot:  int32 a | int32 b   (indices into the blanket's KEPT list, a<b),
 *                double meas[P]      (Z = Xa^-1 Xb, setMeasurementFromState)
 *                double info[d*d]    (X_e, column-major; reference vertex_remover.cpp:531-533)
 *     GLC slot:  int32 nv | int32 rank
 *                int32 vidx[nvcap] (padded)   kept-list indices
 *                double meas[d*nvcap]
 *                double W[d*nvcap][d*nvcap]   row-major, rows >= rank are zero, Omega = I_rank
 *       nvcap = 2 for Tree, n_kept for Dense.
 */

#define SPG_REC_HEADER_WORDS 4
#define SPG_OUT_HEADER_WORDS 4

typedef struct {
    int32_t dim;                 /* 3 | 6                                                   */
    int32_t algorithm;           /* spg_algorithm                                           */
    spg_sparsity_options opts;
    int32_t n_blankets;
    int32_t reserved;
    const int64_t *rec_off;      /* [n_blankets+1] word offsets into records                */
    const uint64_t *records;     /* packed input records                                    */
    const int64_t *out_off;      /* [n_blankets+1] word offsets into out                    */
} spg_round_in;

typedef struct {
    uint64_t *out;               /* packed output records, out_off[n_blankets] words        */
    double *dbg_target;          /* optional: Lambda_t of every blanket, k*k each, packed   */
    const int64_t *dbg_target_off; /* [n_blankets+1] offsets (doubles) into dbg_target, or NULL */
    double *dbg_weights;         /* optional: Chow-Liu MI weights, pairs in (i<j) lexicographic order */
    const int64_t *dbg_weights_off;
} spg_round_out;

typedef struct {
    int32_t device;              /* CUDA device ordinal                                      */
    int32_t reserved;
    int64_t max_record_words;    /* initial device buffer sizes (grown on demand)            */
    int64_t max_out_words;
} spg_config;

typedef struct spg_ctx spg_ctx;

/* library / context */
const char *spg_version(void);
const char *spg_last_error(void);
spg_status spg_create(spg_ctx **ctx, const spg_config *cfg);
void spg_destroy(spg_ctx *ctx);
/* grow the context's page-locked staging buffers (round records / round outputs of the graph level) ahead of time:
 * page-locking hundreds of MB costs tenths of a second, better spent outside a latency-sensitive removal */
spg_status spg_reserve_staging(spg_ctx *ctx, int64_t record_words, int64_t out_words);
/* number of kernels launched by this context so far (bench.py's gpu_launches) */
int64_t spg_launch_count(const spg_ctx *ctx);
/* device time (ms, CUDA events on the context stream) of the kernels of the last round */
double spg_last_kernel_ms(const spg_ctx *ctx);
/* diagnostics: blankets of the last spg_remove_round* call that the NFR-tree kernel (fast_kernel) handed over to the
 * general blanket_kernel (GLC / MULTI edges, several removed vertices, refused gauge guard); synchronises */
int64_t spg_last_retry_count(spg_ctx *ctx);

/* record sizing + packing helpers (pure host code, usable without a GPU) */
int64_t spg_pose_words(int32_t dim);                       /* 3 or 7 */
int64_t spg_record_words(int32_t dim, int32_t n_vert, int32_t n_edges,
                         const int32_t *edge_kind, const int32_t *edge_nv,
                         const int32_t *edge_rows);
int64_t spg_out_record_words(int32_t dim, int32_t algorithm, const spg_sparsity_options *opts,
                             int32_t n_kept);
int32_t spg_out_edge_count(int32_t algorithm, const spg_sparsity_options *opts, int32_t n_kept);
int64_t spg_out_slot_words(int32_t dim, int32_t algorithm, const spg_sparsity_options *opts,
                           int32_t n_kept);

/*
 * One wavefront round through the GPU, host buffers in and out.
 * Replaces, for every blanket of the round, the body of the loop in
 * VertexRemover::remove (src/vertex_remover.cpp:89-139): computeTargetInformation (:394-450),
 * tp->topology (:111), buildJacobianMapping + optimizeInformation (:123-126).
 * Synchronous: H2D copy, kernels, D2H copy, stream sync.
 */
spg_status spg_remove_round(spg_ctx *ctx, const spg_round_in *in, spg_round_out *out);

/*
 * The same call with the records produced on demand: `in->rec_off` / `in->out_off` are complete, `in->records` points at
 * a buffer of rec_off[n_blankets] words that `fill(user, b0, b1)` fills for blankets [b0, b1) (return 0; anything else
 * aborts with SPG_ERR_INVALID). fill is called once per pipeline chunk, in order, on the calling thread, right before
 * the chunk is validated and copied — so packing chunk c+1 overlaps the GPU work on chunk c. A VertexRemover adapter
 * packs straight from its graph structures this way (spg_graph_marginalize does). Page-locked buffers make the copies
 * asynchronous.
 */
typedef int32_t (*spg_fill_fn)(void *user, int32_t first_blanket, int32_t end_blanket);
spg_status spg_remove_round_streamed(spg_ctx *ctx, const spg_round_in *in, spg_round_out *out, spg_fill_fn fill, void *user);

/*
 * Both ends on demand: as above (fill may be NULL: the records are there already), and `drain(user, b0, b1)` is called on
 * the calling thread once the output records of blankets [b0, b1) are complete in out->out — per pipeline chunk, in
 * order, each chunk exactly once: between two fills when a chunk happens to be back, and one by one after the last
 * fill. A VertexRemover adapter splices chunk c into its graph (updateInputGraph, src/vertex_remover.cpp:500-546)
 * while the GPU works on the chunks behind it, instead of waiting for the whole round (spg_graph_marginalize does; the
 * blankets of a round commute, so splicing some while others are still being packed is safe as long as packing reads
 * nothing but its own blanket). A nonzero return aborts with SPG_ERR_INVALID.
 */
typedef int32_t (*spg_drain_fn)(void *user, int32_t first_blanket, int32_t end_blanket);
spg_status spg_remove_round_pipelined(spg_ctx *ctx, const spg_round_in *in, spg_round_out *out, spg_fill_fn fill, spg_drain_fn drain,
                                      void *user);

/*
 * Same, but every pointer inside in/out is a DEVICE pointer already resident in HBM
 * (rec_off/out_off too). Asynchronous on the context stream; call spg_sync().
 * The records cannot be validated from the host here: the caller states the largest blanket of the round
 * (vertices, edges, record words; max_rec_words = 0 means "POSE edges only": the bound is derived). A record
 * beyond these bounds is answered with SPG_BLANKET_TOO_LARGE; the records themselves must be well formed
 * (spg_remove_round checks that on the host for host buffers).
 */
spg_status spg_remove_round_device(spg_ctx *ctx, const spg_round_in *in_dev, spg_round_out *out_dev,
                                   int32_t max_n_vert, int32_t max_n_edges, int32_t max_rec_words);
spg_status spg_sync(spg_ctx *ctx);
void *spg_stream(spg_ctx *ctx); /* cudaStream_t of the context */

/* ------------------------------------------------------------------------------------------ */
/* Sharded rounds: one process per GPU, the blankets of a round split over the ranks          */
/* ------------------------------------------------------------------------------------------ */
/*
 * The reference is single-threaded (src/evaluate.cpp:342-411 runs one job per process); SURVEY §8(e) shards the
 * independent blankets of a wavefront round over the GPUs of a box. Every rank holds the same round description
 * (the graph is replicated or lives on the root), runs a contiguous cost-balanced shard on its GPU, and the
 * substitute-edge records are gathered with NCCL over NVLink directly between the device output buffers
 * (ragged all-gather, or send/recv to `root`). NCCL is bound with dlopen at spg_comm_init: the library has no
 * link-time dependency on it.
 *   rank 0: spg_comm_unique_id(id); ...ship id to the other ranks (MPI, torch.distributed, a file)...
 *   all   : spg_comm_init(ctx, nranks, rank, id);   (nranks == 1 is valid and needs no NCCL)
 */
#define SPG_COMM_ID_BYTES 128
spg_status spg_comm_unique_id(uint8_t *id /* SPG_COMM_ID_BYTES */);
spg_status spg_comm_init(spg_ctx *ctx, int32_t nranks, int32_t rank, const uint8_t *id);
spg_status spg_comm_destroy(spg_ctx *ctx);
int32_t spg_comm_nranks(const spg_ctx *ctx);
int32_t spg_comm_rank(const spg_ctx *ctx);
int32_t spg_comm_nccl_version(void); /* 0: NCCL not loadable */

/* contiguous shards of a round balanced by a per-blanket cost model (cubic in the blanket size):
 * bounds[r] .. bounds[r+1] is rank r's part. Pure host code. */
spg_status spg_shard_bounds(const spg_round_in *in, int32_t nranks, int32_t *bounds /* nranks+1 */);

typedef struct {
    int32_t nranks, rank;
    int32_t n_blankets_mine, reserved0; /* blankets this rank ran                                   */
    int32_t steps, reserved;            /* pipeline steps (H2D | kernels | gather | D2H overlap)    */
    double kernel_ms;                   /* first to last kernel of this rank                        */
    double gather_window_ms;            /* first to last gather on the gather stream (overlaps)     */
    int64_t gather_bytes;               /* bytes this rank sent or received over NVLink             */
    int64_t h2d_bytes, d2h_bytes;       /* bytes this rank copied host -> device / device -> host   */
} spg_shard_info;

/*
 * spg_remove_round over all ranks of the communicator. Collective: every rank calls it with the SAME round (host
 * buffers; a rank only reads the records of its own blankets, and the headers of the others for the balance).
 * The round is cut into pipeline steps of about equal bytes and every step is split over the ranks by bytes again
 * (offset tables only: the plan is derived by every rank on every call and must not touch the records), so each rank
 * moves 1/nranks of the bytes of every step and — cost per byte being flat within a step — does 1/nranks of its work.
 * root == -1: every rank gets the complete output (replicated graphs, all-gather); root >= 0: only that rank does
 * (the others get the records of their own blankets). root == SPG_ROOT_SHARED_HOST: no device gather at all — `out->out`
 * is ONE host buffer mapped by every rank of the box (POSIX shared memory, page-locked in each process) and every rank
 * copies the records of its own blankets straight into it over its own PCIe link; the caller synchronises the ranks
 * before the graph-holding process reads the buffer. That is the fastest way to a host-resident graph on one node (the
 * root of a gather is bound by ITS device -> host copy of everything); the NCCL modes serve device-resident consumers
 * and replicated graphs. info may be NULL.
 */
#define SPG_ROOT_SHARED_HOST (-2)
spg_status spg_remove_round_sharded(spg_ctx *ctx, const spg_round_in *in, spg_round_out *out, int32_t root,
                                    spg_shard_info *info);
/*
 * Device-resident variant (asynchronous; spg_sync() also drains the gather stream): in_dev / out_dev describe the
 * whole round in HBM at identical offsets on every rank; the caller gives the shard bounds (blankets) and the
 * matching word offsets into out (both nranks+1 host arrays). The gather of this call overlaps the kernels of
 * the next one.
 */
spg_status spg_remove_round_sharded_device(spg_ctx *ctx, const spg_round_in *in_dev, spg_round_out *out_dev,
                                           const int32_t *bounds, const int64_t *out_word_bounds,
                                           int32_t max_n_vert, int32_t max_n_edges, int32_t max_rec_words,
                                           int32_t root);

/* the context stream waits (on the device, asynchronously) for every gather issued so far: call it before the output
 * buffers of a spg_remove_round_sharded_device call are read by later work on spg_stream() or written again */
spg_status spg_comm_join(spg_ctx *ctx);

/*
 * Roofline denominator: register-resident DFMA loop on every SM (no memory traffic), timed with
 * CUDA events. MEASURED_PEAKS.json carries no FP64 figure, so bench.py measures it with this.
 * Returns the best of `repeats` in TFLOP/s (2 flops per DFMA).
 */
spg_status spg_fp64_peak_probe(spg_ctx *ctx, int32_t repeats, double *tflops);
/* developer aid: per-stage clock64() accumulators of the fused kernel (16 values), see tools/stage_profile.py */
spg_status spg_stage_profile(spg_ctx *ctx, int32_t enable, uint64_t *cycles);

/* ------------------------------------------------------------------------------------------ */
/* Graph level: g2o-free container with the reference's removal semantics.                    */
/* Mirrors GraphWrapper (src/graph_wrapper.h:17-81) for the calls on the removal path.        */
/* ------------------------------------------------------------------------------------------ */

typedef struct spg_graph spg_graph;

spg_status spg_graph_create(spg_graph **g, int32_t dim);
void spg_graph_destroy(spg_graph *g);
/* reads VERTEX_SE2/EDGE_SE2/VERTEX_SE3:QUAT/EDGE_SE3:QUAT (src/graph_wrapper_g2o.cpp:107-147) and the factor types of
 * a saved sparsified graph: EDGE_SE2_ISAM, GLC_EDGE with GLC_REPARAM_{SE2_ISAM,SE2,SE3} (src/glc_edge.cpp:64-118),
 * MULTI_EDGE_{SE2,SE2_ISAM,SE3,SE3_ISAM} (src/multi_edge_correlated.hpp:183-267; tags src/edge_types.cpp:68-76) */
spg_status spg_graph_load_g2o(spg_graph **g, const char *path);
/* GraphWrapperG2O::write (src/graph_wrapper_g2o.cpp:467-470): the same text format, 17 significant digits. A multi-edge
 * is preceded by a comment line "#SPG_MULTI_PAIRS .." with the vertex pair of every measurement (the reference's
 * format drops them; stock g2o skips comment lines). */
spg_status spg_graph_save_g2o(const spg_graph *g, const char *path);
/* generic factor (an adapter copying GLCEdge / MultiEdgeCorrelated objects out of g2o): kind = spg_edge_kind;
 * POSE: nv 2, rows d, meas P, info d*d column-major; GLC: meas d*nv, W rows x d*nv row-major; MULTI: rows = d*nmeas,
 * meas nmeas*P, info rows*rows column-major, pairs = 2*nmeas indices into vert_ids (NULL otherwise) */
spg_status spg_graph_add_factor(spg_graph *g, int32_t kind, int32_t nv, const int32_t *vert_ids, int32_t rows,
                                const double *meas, const double *info_or_w, const int32_t *pairs);
/* MULTI edges: the 2*nmeas vertex-list indices of the measurements (see spg_graph_edge_desc for sizes) */
spg_status spg_graph_edge_pairs(const spg_graph *g, int32_t idx, int32_t *pairs);
spg_status spg_graph_add_vertex(spg_graph *g, int32_t id, const double *pose);
spg_status spg_graph_add_edge(spg_graph *g, int32_t from, int32_t to, const double *meas,
                              const double *info /* d*d column-major */);
int32_t spg_graph_dim(const spg_graph *g);
int32_t spg_graph_num_vertices(const spg_graph *g);
int32_t spg_graph_num_edges(const spg_graph *g);
int32_t spg_graph_max_vertex_id(const spg_graph *g);

/* removal schedules, reference src/decimation.cpp:11-49. Returns count; ids written to out (cap).
 * sparsity <= 0 (or cluster_size <= 0) would divide by zero in the reference: returns -1. */
int32_t spg_decimate_global(int32_t last, int32_t endvert, int32_t sparsity, int32_t *out, int32_t cap);
int32_t spg_decimate_online(int32_t last, int32_t endvert, int32_t sparsity, int32_t *out, int32_t cap);
int32_t spg_decimate_cluster(int32_t last, int32_t endvert, int32_t sparsity, int32_t cluster_size,
                             int32_t *out, int32_t cap);

/*
 * GraphWrapperG2O::marginalizeNoOptimize(which, options) (src/graph_wrapper_g2o.cpp:398-453):
 * removes the vertices `which` (in this order) and splices the substitute edges in. The result is
 * identical to the reference's one-at-a-time loop; internally removals are grouped into
 * wavefront rounds of non-interfering blankets, each round is one spg_remove_round().
 * With a communicator on ctx (spg_comm_init, nranks > 1) the call is collective: every rank passes an identical
 * graph and list, each round is one spg_remove_round_sharded(root = -1), and the graphs stay identical.
 */
spg_status spg_graph_marginalize(spg_graph *g, spg_ctx *ctx, const int32_t *which, int32_t n_which,
                                 const spg_sparsity_options *opts, int32_t algorithm);

/*
 * The same removal, one wavefront round at a time, for callers that run the blankets of a round
 * themselves (sharded over ranks / GPUs):
 *   spg_graph_rounds_begin(g, which, n, opts, alg);
 *   for (;;) { spg_graph_round_next(g, &round); if (round.n_blankets == 0) break;
 *              ... fill `out` (round.out_off[n_blankets] words) with spg_remove_round on any split ...
 *              spg_graph_round_apply(g, out); }
 * The pointers inside `round` stay valid until the next spg_graph_round_* call.
 */
spg_status spg_graph_rounds_begin(spg_graph *g, const int32_t *which, int32_t n_which,
                                  const spg_sparsity_options *opts, int32_t algorithm);
spg_status spg_graph_round_next(spg_graph *g, spg_round_in *round);
spg_status spg_graph_round_apply(spg_graph *g, const uint64_t *out);

typedef struct {
    int32_t n_rounds;
    int32_t n_blankets;
    int32_t max_round_width;
    int32_t max_blanket_vertices;
    int32_t n_failed;            /* blankets whose status != OK: left in the graph, call returns SPG_ERR_BLANKET_FAILED */
    int32_t n_dropped_edges;     /* GLC rank-0 edges (reference returns NULL, :85-89) */
    double pack_ms, gpu_ms, splice_ms;
    int32_t first_failed_index;  /* index into `which` of the first failed blanket, -1 if none */
    int32_t first_failed_status; /* its spg_blanket_status */
    int32_t n_applied;           /* list entries whose removal was spliced into the graph (progress on error) */
    int32_t n_local_optimised;   /* Local lin. point: non-star blankets whose subgraph was optimised (:382-391) */
} spg_marginalize_stats;
spg_status spg_graph_last_stats(const spg_graph *g, spg_marginalize_stats *stats);

/* read-back of the current edge list (for parity tests / writers). Edge index order is the
 * canonical creation order. */
typedef struct {
    int32_t kind;      /* spg_edge_kind */
    int32_t nv;
    int32_t rows;
    int32_t uid_major; /* -1 for file edges, else index in the removal list that created it */
    int32_t uid_minor; /* file order / provider order */
} spg_edge_desc;
spg_status spg_graph_edge_desc(const spg_graph *g, int32_t idx, spg_edge_desc *desc);
/* vertex ids (nv), measurement (P or d*nv doubles), info-or-W (d*d col-major, or rows*d*nv row-major) */
spg_status spg_graph_edge_data(const spg_graph *g, int32_t idx, int32_t *vert_ids, double *meas,
                               double *info_or_w);
spg_status spg_graph_vertex_ids(const spg_graph *g, int32_t *ids /* num_vertices */);
spg_status spg_graph_vertex_pose(const spg_graph *g, int32_t id, double *pose);

/* ------------------------------------------------------------------------------------------ */
/* Whole-graph evaluator and optimiser on the GPU (the steps either side of the removal path) */
/* ------------------------------------------------------------------------------------------ */
typedef struct {
    double innerprod;      /* tr(Lambda_y^-1 Lambda_x)                                        */
    double mahalanobis;    /* d^T Lambda_x d, d = estimateDifference                          */
    double logdet_x;       /* sparsified graph                                                */
    double logdet_y;       /* true marginal of the full graph                                 */
    int32_t n_keep;        /* dimensions both informations have                               */
    int32_t n_marginalized;
    double device_ms;      /* assembly + factorisations, CUDA events                          */
    double flops;          /* dense flops of the factorisations / solves (n^3/3 conventions)  */
} spg_kld_terms;
/*
 * GraphWrapperG2O::kullbackLeibler(other) (src/graph_wrapper_g2o.cpp:531-548, src/utils.cpp:70-97, mode
 * InformationInformation): `full` is the unsparsified graph, `sparse` the sparsified one (its vertices are a subset).
 * Both informations are H = sum J^T Omega J at the graphs' current estimates with vertex `fixed_id` (0 in the
 * reference) held fixed; the full graph's is marginalised onto the kept variables by a partial blocked Cholesky.
 * POSE and GLC factors. terms may be NULL.
 */
spg_status spg_graph_kld(spg_ctx *ctx, const spg_graph *full, const spg_graph *sparse, int32_t fixed_id, double *kld,
                         spg_kld_terms *terms);

typedef struct {
    int32_t iterations;    /* outer Levenberg-Marquardt iterations run                        */
    int32_t trials;        /* linear solves (an iteration retries with a larger lambda)       */
    int32_t dimensions;
    int32_t terminated;    /* 1: g2o's Terminate (no acceptable step), 0: iteration limit     */
    double chi2_initial, chi2_final, lambda_final;
    int32_t solver;        /* SPG_SOLVER_DENSE_CHOLESKY or SPG_SOLVER_SPARSE_PCG                */
    int32_t cg_iterations; /* PCG iterations summed over all trials (0 on the dense path)        */
    double cg_max_rel_residual; /* largest ||r|| / ||b|| at which a trial's PCG stopped          */
} spg_optimize_stats;
#define SPG_SOLVER_DENSE_CHOLESKY 0
#define SPG_SOLVER_SPARSE_PCG 1
/*
 * GraphWrapperG2O::optimize (src/graph_wrapper_g2o.cpp:250-269): g2o's OptimizationAlgorithmLevenberg with its
 * default parameters (tau 1e-5, step scales 1/3 .. 2/3, 10 trials after a failure), max_iterations = 50 in the
 * reference, the listed vertices fixed (the reference fixes vertex 0). The estimates of the graph are updated in place.
 * stats may be NULL.
 * The linear system (H + lambda I) x = -g is solved one of two ways, chosen from the problem size and free device
 * memory alone:
 *   - dense (SPG_SOLVER_DENSE_CHOLESKY): H assembled dense in HBM and factorised by a blocked Cholesky, whenever
 *     n^2 * 8 <= 120e9 bytes (n = free dimensions, ~122 k) and the two n x n buffers can be allocated;
 *   - block-sparse (SPG_SOLVER_SPARSE_PCG): otherwise. H in BSR (D x D blocks of both triangles) and solved by
 *     conjugate gradients with a block-Jacobi preconditioner (g2o's LinearSolverPCG), from x = 0 to
 *     ||r|| <= 1e-6 ||b|| or 5000 iterations; a trial that reaches the cap still proposes its step to the rho test.
 * The environment variable SPG_OPT_DENSE_MAX_DIMS (read on every call) lowers the dense path's limit to that many
 * dimensions; it exists for tests, like SPG_CHUNK_BYTES.
 */
spg_status spg_graph_optimize(spg_ctx *ctx, spg_graph *g, const int32_t *fixed_ids, int32_t n_fixed, int32_t max_iterations,
                              spg_optimize_stats *stats);
/* OptimizableGraph::chi2 at the current estimates: sum e^T Omega e over all factors */
spg_status spg_graph_chi2(spg_ctx *ctx, const spg_graph *g, double *chi2);
/* overwrite the estimate of a vertex (GraphWrapper::setEstimate) */
spg_status spg_graph_set_vertex_pose(spg_graph *g, int32_t id, const double *pose);

/* ------------------------------------------------------------------------------------------ */
/* evaluate(): the replay loop of the reference's `sparsifier` binary                         */
/* ------------------------------------------------------------------------------------------ */
#define SPG_EVAL_NONE (-1)    /* EvaluateInfo::None: no sparsification, baseline only */
typedef enum { SPG_PROFILE_ONLINE = 0, SPG_PROFILE_CLUSTER = 1, SPG_PROFILE_GLOBAL = 2 } spg_profile; /* decimation.cpp */
/* EvaluateInfo (src/evaluate.h:16-31) */
typedef struct {
    int32_t algorithm;          /* SPG_ALG_NFR | SPG_ALG_GLC | SPG_EVAL_NONE                          */
    int32_t profile;            /* spg_profile: which decimate function                              */
    spg_sparsity_options opts;
    int32_t sparsity, cluster_size;
    int32_t kld_period;
    int32_t use_chi2;           /* delta chi2 instead of the KLD                                      */
    const char *g2oname;        /* names the result files (may be NULL)                               */
    const char *destdir;        /* NULL: no result files; else <destdir>/<profile>/<sparsity>/<dataset>/<alg>_<type>_<l|g>.{kld,txt} */
} spg_evaluate_info;
typedef struct {
    int32_t n_samples;          /* KLD / chi2 samples taken (may exceed the caller's capacity)        */
    int32_t last_vertex;
    double last_value;
    int32_t baseline_nodes, baseline_edges, marginal_nodes, marginal_edges; /* printStats (:606-612) */
    double baseline_fillin, marginal_fillin;
    double seconds_marginalize, seconds_optimize, seconds_kld;
    int32_t n_marginalize_calls, n_marginalized;
} spg_evaluate_result;
/* parseLine (src/main.cpp:9-103): one job line "<nfr|glc|none> <file.g2o> <online|cluster|global>
 * <tree|subgr|clsubgr|dense|cldense> <local|global> <sparsity> [kldPeriod [chi2|kld [clusterSize]]]";
 * the file name is copied to g2oname (cap bytes) and info->g2oname points at it */
spg_status spg_evaluate_parse_job(const char *line, spg_evaluate_info *info, char *g2oname, int32_t cap);
/*
 * evaluate(gw, info) (src/evaluate.cpp:32-221): grows an incremental and a baseline graph from `gw` vertex by vertex
 * (ids 0..last must exist), links to already-marginalised vertices through computeSubstituteEdge, optimises both,
 * marginalises the incremental one on the decimation schedule (spg_graph_marginalize + optimise) and samples
 * KLD(baseline || incremental) — or the delta chi2 — every kld_period vertices and at the end. Samples go to
 * sample_vertex / sample_value (cap entries; may be NULL) and, with destdir, to the reference's result files.
 * incremental_out / baseline_out (may be NULL) receive the final graphs (spg_graph_destroy them).
 */
spg_status spg_evaluate(spg_ctx *ctx, const spg_graph *gw, const spg_evaluate_info *info, int32_t *sample_vertex,
                        double *sample_value, int32_t cap, spg_evaluate_result *res, spg_graph **incremental_out,
                        spg_graph **baseline_out);

/*
 * computeSubstituteEdge (src/compute_substitute_edge.cpp:13-96) on this container.
 * marginalized: sorted ids. from/to are in-out. meas: P doubles, info: d*d column-major.
 */
spg_status spg_compute_substitute_edge(const spg_graph *g, const int32_t *marginalized,
                                       int32_t n_marginalized, int32_t maxid, int32_t *from,
                                       int32_t *to, double *meas, double *info);

#ifdef __cplusplus
}
#endif
#endif /* SPG_CAPI_H_ */
