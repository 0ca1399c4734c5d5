"""ctypes binding of libspg_b200.so (include/spg_capi.h).

The CUDA library is the product; this module only marshals numpy buffers / raw device pointers
into the C ABI. There is no CPU implementation behind it: if the shared library is missing or no
sm_100 device is present, calls raise.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SPG_LIB") or os.path.join(_HERE, "libspg_b200.so")


class SparsityOptions(C.Structure):
    """reference src/sparsity_options.h:11-30"""
    _fields_ = [("topology", C.c_int32), ("lin_point", C.c_int32), ("chord_ratio", C.c_double),
                ("include_intra_clique", C.c_int32), ("reserved", C.c_int32)]


class RoundIn(C.Structure):
    _fields_ = [("dim", C.c_int32), ("algorithm", C.c_int32), ("opts", SparsityOptions),
                ("n_blankets", C.c_int32), ("reserved", C.c_int32),
                ("rec_off", C.c_void_p), ("records", C.c_void_p), ("out_off", C.c_void_p)]


class RoundOut(C.Structure):
    _fields_ = [("out", C.c_void_p), ("dbg_target", C.c_void_p), ("dbg_target_off", C.c_void_p),
                ("dbg_weights", C.c_void_p), ("dbg_weights_off", C.c_void_p)]


class Config(C.Structure):
    _fields_ = [("device", C.c_int32), ("reserved", C.c_int32), ("max_record_words", C.c_int64),
                ("max_out_words", C.c_int64)]


class EdgeDesc(C.Structure):
    _fields_ = [("kind", C.c_int32), ("nv", C.c_int32), ("rows", C.c_int32), ("uid_major", C.c_int32),
                ("uid_minor", C.c_int32)]


class MarginalizeStats(C.Structure):
    _fields_ = [("n_rounds", C.c_int32), ("n_blankets", C.c_int32), ("max_round_width", C.c_int32),
                ("max_blanket_vertices", C.c_int32), ("n_failed", C.c_int32), ("n_dropped_edges", C.c_int32),
                ("pack_ms", C.c_double), ("gpu_ms", C.c_double), ("splice_ms", C.c_double),
                ("first_failed_index", C.c_int32), ("first_failed_status", C.c_int32), ("n_applied", C.c_int32),
                ("n_local_optimised", C.c_int32)]


class ShardInfo(C.Structure):
    _fields_ = [("nranks", C.c_int32), ("rank", C.c_int32), ("n_blankets_mine", C.c_int32), ("reserved0", C.c_int32),
                ("steps", C.c_int32), ("reserved", C.c_int32), ("kernel_ms", C.c_double), ("gather_window_ms", C.c_double),
                ("gather_bytes", C.c_int64), ("h2d_bytes", C.c_int64), ("d2h_bytes", C.c_int64)]


COMM_ID_BYTES = 128


class KldTerms(C.Structure):
    _fields_ = [("innerprod", C.c_double), ("mahalanobis", C.c_double), ("logdet_x", C.c_double), ("logdet_y", C.c_double),
                ("n_keep", C.c_int32), ("n_marginalized", C.c_int32), ("device_ms", C.c_double), ("flops", C.c_double)]


class OptimizeStats(C.Structure):
    _fields_ = [("iterations", C.c_int32), ("trials", C.c_int32), ("dimensions", C.c_int32), ("terminated", C.c_int32),
                ("chi2_initial", C.c_double), ("chi2_final", C.c_double), ("lambda_final", C.c_double),
                ("solver", C.c_int32), ("cg_iterations", C.c_int32), ("cg_max_rel_residual", C.c_double)]


SOLVER_DENSE_CHOLESKY, SOLVER_SPARSE_PCG = 0, 1   # OptimizeStats.solver


class EvaluateInfo(C.Structure):
    """EvaluateInfo, reference src/evaluate.h:16-31"""
    _fields_ = [("algorithm", C.c_int32), ("profile", C.c_int32), ("opts", SparsityOptions), ("sparsity", C.c_int32),
                ("cluster_size", C.c_int32), ("kld_period", C.c_int32), ("use_chi2", C.c_int32), ("g2oname", C.c_char_p),
                ("destdir", C.c_char_p)]


class EvaluateResult(C.Structure):
    _fields_ = [("n_samples", C.c_int32), ("last_vertex", C.c_int32), ("last_value", C.c_double), ("baseline_nodes", C.c_int32),
                ("baseline_edges", C.c_int32), ("marginal_nodes", C.c_int32), ("marginal_edges", C.c_int32),
                ("baseline_fillin", C.c_double), ("marginal_fillin", C.c_double), ("seconds_marginalize", C.c_double),
                ("seconds_optimize", C.c_double), ("seconds_kld", C.c_double), ("n_marginalize_calls", C.c_int32),
                ("n_marginalized", C.c_int32)]


class SpgError(RuntimeError):
    pass


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise SpgError(f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(there is no CPU fallback for the node-removal path)")
        L = C.CDLL(LIB_PATH)
        L.spg_version.restype = C.c_char_p
        L.spg_last_error.restype = C.c_char_p
        L.spg_create.argtypes = [C.POINTER(C.c_void_p), C.POINTER(Config)]
        L.spg_destroy.argtypes = [C.c_void_p]
        L.spg_launch_count.restype = C.c_int64
        L.spg_launch_count.argtypes = [C.c_void_p]
        L.spg_last_kernel_ms.restype = C.c_double
        L.spg_last_kernel_ms.argtypes = [C.c_void_p]
        L.spg_last_retry_count.restype = C.c_int64
        L.spg_last_retry_count.argtypes = [C.c_void_p]
        L.spg_remove_round.argtypes = [C.c_void_p, C.POINTER(RoundIn), C.POINTER(RoundOut)]
        L.spg_remove_round_device.argtypes = [C.c_void_p, C.POINTER(RoundIn), C.POINTER(RoundOut), C.c_int32, C.c_int32, C.c_int32]
        L.spg_sync.argtypes = [C.c_void_p]
        L.spg_stream.restype = C.c_void_p
        L.spg_stream.argtypes = [C.c_void_p]
        L.spg_out_record_words.restype = C.c_int64
        L.spg_out_record_words.argtypes = [C.c_int32, C.c_int32, C.POINTER(SparsityOptions), C.c_int32]
        L.spg_fp64_peak_probe.argtypes = [C.c_void_p, C.c_int32, C.POINTER(C.c_double)]
        L.spg_comm_unique_id.argtypes = [C.c_void_p]
        L.spg_comm_init.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p]
        L.spg_comm_destroy.argtypes = [C.c_void_p]
        L.spg_comm_join.argtypes = [C.c_void_p]
        L.spg_comm_nranks.argtypes = [C.c_void_p]
        L.spg_comm_rank.argtypes = [C.c_void_p]
        L.spg_shard_bounds.argtypes = [C.POINTER(RoundIn), C.c_int32, C.c_void_p]
        L.spg_remove_round_sharded.argtypes = [C.c_void_p, C.POINTER(RoundIn), C.POINTER(RoundOut), C.c_int32, C.POINTER(ShardInfo)]
        L.spg_remove_round_sharded_device.argtypes = [C.c_void_p, C.POINTER(RoundIn), C.POINTER(RoundOut), C.c_void_p, C.c_void_p,
                                                      C.c_int32, C.c_int32, C.c_int32, C.c_int32]
        _lib = L
    return _lib


def make_opts(topology=0, lin_point=1, chord_ratio=1.0, include_intra_clique=True, flags=0):
    return SparsityOptions(int(topology), int(lin_point), float(chord_ratio), int(bool(include_intra_clique)), int(flags))


def _check(rc):
    if rc != 0:
        raise SpgError(f"spg status {rc}: {lib().spg_last_error().decode()}")


def _p(a):
    return a.ctypes.data_as(C.c_void_p).value if a is not None else None


class Context:
    """spg_ctx: one CUDA device, one stream, growable device staging buffers."""

    def __init__(self, device=0):
        self.h = C.c_void_p()
        cfg = Config(int(device), 0, 0, 0)
        _check(lib().spg_create(C.byref(self.h), C.byref(cfg)))

    def close(self):
        if getattr(self, "h", None):
            lib().spg_destroy(self.h)
            self.h = None

    def __del__(self):
        self.close()

    @property
    def launches(self):
        return int(lib().spg_launch_count(self.h))

    @property
    def last_kernel_ms(self):
        return float(lib().spg_last_kernel_ms(self.h))

    @property
    def last_retry_count(self):
        return int(lib().spg_last_retry_count(self.h))

    def stream(self):
        return lib().spg_stream(self.h)

    def remove_round(self, dim, algorithm, opts, records, rec_off, out_off, out=None, want_target=None,
                     want_weights=None, weights_in=None):
        """Host buffers in / out (H2D + kernels + D2H inside). Returns (out, dbg_target, dbg_weights).
        weights_in (with opts.flags & SPG_OPT_DBG_WEIGHTS_IN and want_weights offsets): test hook, see spg_capi.h."""
        records = np.ascontiguousarray(records, dtype=np.uint64)
        rec_off = np.ascontiguousarray(rec_off, dtype=np.int64)
        out_off = np.ascontiguousarray(out_off, dtype=np.int64)
        nb = len(rec_off) - 1
        if out is None:
            out = np.empty(int(out_off[-1]), dtype=np.uint64)
        rin = RoundIn(dim, algorithm, opts, nb, 0, _p(rec_off), _p(records), _p(out_off))
        rout = RoundOut(_p(out), None, None, None, None)
        tgt = wts = None
        if want_target is not None:
            want_target = np.ascontiguousarray(want_target, dtype=np.int64)
            tgt = np.zeros(int(want_target[-1]), dtype=np.float64)
            rout.dbg_target, rout.dbg_target_off = _p(tgt), _p(want_target)
        if want_weights is not None:
            want_weights = np.ascontiguousarray(want_weights, dtype=np.int64)
            wts = np.zeros(int(want_weights[-1]), dtype=np.float64)
            if weights_in is not None:
                wts[:] = weights_in
            rout.dbg_weights, rout.dbg_weights_off = _p(wts), _p(want_weights)
        _check(lib().spg_remove_round(self.h, C.byref(rin), C.byref(rout)))
        return out, tgt, wts

    def remove_round_device(self, dim, algorithm, opts, n_blankets, d_records, d_rec_off, d_out_off, d_out,
                            max_n_vert, max_n_edges, max_rec_words=0):
        """Device pointers (ints) already resident in HBM; asynchronous on the context stream."""
        rin = RoundIn(dim, algorithm, opts, int(n_blankets), 0, int(d_rec_off), int(d_records), int(d_out_off))
        rout = RoundOut(int(d_out), None, None, None, None)
        _check(lib().spg_remove_round_device(self.h, C.byref(rin), C.byref(rout), int(max_n_vert), int(max_n_edges),
                                                 int(max_rec_words)))

    def sync(self):
        _check(lib().spg_sync(self.h))

    def reserve_staging(self, record_words, out_words):
        """Page-lock the graph-level staging buffers ahead of time (spg_reserve_staging)."""
        L = lib()
        L.spg_reserve_staging.argtypes = [C.c_void_p, C.c_int64, C.c_int64]
        _check(L.spg_reserve_staging(self.h, int(record_words), int(out_words)))

    # ---- sharded rounds (spg_comm.cu): one process per GPU, NCCL gather of the substitute-edge records -------------
    def comm_init(self, nranks, rank, unique_id=None):
        """unique_id: the SPG_COMM_ID_BYTES bytes rank 0 got from comm_unique_id() (any transport); None for nranks == 1."""
        buf = None
        if unique_id is not None:
            buf = np.frombuffer(bytes(unique_id), dtype=np.uint8).copy()
            assert len(buf) == COMM_ID_BYTES
        _check(lib().spg_comm_init(self.h, int(nranks), int(rank), _p(buf)))

    def comm_join(self):
        """The context stream waits for the gathers issued so far (asynchronous)."""
        _check(lib().spg_comm_join(self.h))

    def comm_destroy(self):
        _check(lib().spg_comm_destroy(self.h))

    @property
    def nranks(self):
        return int(lib().spg_comm_nranks(self.h))

    @property
    def rank(self):
        return int(lib().spg_comm_rank(self.h))

    def remove_round_sharded(self, dim, algorithm, opts, records, rec_off, out_off, out=None, root=-1):
        """Collective: the same round on every rank, each runs its shard, outputs gathered over NCCL.
        Returns (out, info dict). root < 0: every rank gets the whole output."""
        records = np.ascontiguousarray(records, dtype=np.uint64)
        rec_off = np.ascontiguousarray(rec_off, dtype=np.int64)
        out_off = np.ascontiguousarray(out_off, dtype=np.int64)
        nb = len(rec_off) - 1
        if out is None:
            out = np.zeros(int(out_off[-1]), dtype=np.uint64)
        rin = RoundIn(dim, algorithm, opts, nb, 0, _p(rec_off), _p(records), _p(out_off))
        rout = RoundOut(_p(out), None, None, None, None)
        info = ShardInfo()
        _check(lib().spg_remove_round_sharded(self.h, C.byref(rin), C.byref(rout), int(root), C.byref(info)))
        return out, {f: getattr(info, f) for f, _ in ShardInfo._fields_}

    def remove_round_sharded_device(self, dim, algorithm, opts, n_blankets, d_records, d_rec_off, d_out_off, d_out, bounds,
                                    out_word_bounds, max_n_vert, max_n_edges, max_rec_words=0, root=-1):
        """Device-resident collective round; bounds / out_word_bounds: nranks+1 host arrays (blankets / output words)."""
        b = np.ascontiguousarray(bounds, dtype=np.int32)
        w = np.ascontiguousarray(out_word_bounds, dtype=np.int64)
        rin = RoundIn(dim, algorithm, opts, int(n_blankets), 0, int(d_rec_off), int(d_records), int(d_out_off))
        rout = RoundOut(int(d_out), None, None, None, None)
        _check(lib().spg_remove_round_sharded_device(self.h, C.byref(rin), C.byref(rout), _p(b), _p(w), int(max_n_vert),
                                                     int(max_n_edges), int(max_rec_words), int(root)))

    def fp64_peak_tflops(self, repeats=5):
        """Measured DFMA peak of this device (roofline denominator for the FP64-bound kernels)."""
        v = C.c_double()
        _check(lib().spg_fp64_peak_probe(self.h, int(repeats), C.byref(v)))
        return float(v.value)


def comm_unique_id():
    """ncclGetUniqueId through the library (rank 0); ship the bytes to the other ranks."""
    buf = np.zeros(COMM_ID_BYTES, dtype=np.uint8)
    _check(lib().spg_comm_unique_id(_p(buf)))
    return buf.tobytes()


def shard_bounds(dim, algorithm, opts, records, rec_off, out_off, nranks):
    """spg_shard_bounds: contiguous cost-balanced shards of a round (pure host code)."""
    records = np.ascontiguousarray(records, dtype=np.uint64)
    rec_off = np.ascontiguousarray(rec_off, dtype=np.int64)
    out_off = np.ascontiguousarray(out_off, dtype=np.int64)
    rin = RoundIn(dim, algorithm, opts, len(rec_off) - 1, 0, _p(rec_off), _p(records), _p(out_off))
    b = np.zeros(nranks + 1, dtype=np.int32)
    _check(lib().spg_shard_bounds(C.byref(rin), int(nranks), _p(b)))
    return b


def _graph_protos(L):
    if getattr(L, "_graph_protos_done", False):
        return
    L.spg_graph_create.argtypes = [C.POINTER(C.c_void_p), C.c_int32]
    L.spg_graph_destroy.argtypes = [C.c_void_p]
    L.spg_graph_load_g2o.argtypes = [C.POINTER(C.c_void_p), C.c_char_p]
    L.spg_graph_save_g2o.argtypes = [C.c_void_p, C.c_char_p]
    L.spg_graph_add_factor.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]
    L.spg_graph_edge_pairs.argtypes = [C.c_void_p, C.c_int32, C.c_void_p]
    L.spg_graph_kld.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.POINTER(C.c_double), C.POINTER(KldTerms)]
    L.spg_graph_optimize.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.POINTER(OptimizeStats)]
    L.spg_graph_chi2.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(C.c_double)]
    L.spg_graph_set_vertex_pose.argtypes = [C.c_void_p, C.c_int32, C.c_void_p]
    L.spg_graph_add_vertex.argtypes = [C.c_void_p, C.c_int32, C.c_void_p]
    L.spg_graph_add_edge.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]
    for f in ("spg_graph_dim", "spg_graph_num_vertices", "spg_graph_num_edges", "spg_graph_max_vertex_id"):
        getattr(L, f).argtypes = [C.c_void_p]
    for f in ("spg_decimate_global", "spg_decimate_online"):
        getattr(L, f).argtypes = [C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_int32]
    L.spg_decimate_cluster.argtypes = [C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_int32]
    L.spg_graph_marginalize.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.POINTER(SparsityOptions), C.c_int32]
    L.spg_graph_last_stats.argtypes = [C.c_void_p, C.POINTER(MarginalizeStats)]
    L.spg_graph_edge_desc.argtypes = [C.c_void_p, C.c_int32, C.POINTER(EdgeDesc)]
    L.spg_graph_edge_data.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]
    L.spg_graph_vertex_ids.argtypes = [C.c_void_p, C.c_void_p]
    L.spg_graph_vertex_pose.argtypes = [C.c_void_p, C.c_int32, C.c_void_p]
    L.spg_compute_substitute_edge.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.POINTER(C.c_int32),
                                              C.POINTER(C.c_int32), C.c_void_p, C.c_void_p]
    L._graph_protos_done = True


class Graph:
    """spg_graph: g2o-free pose graph with the reference's removal semantics
    (GraphWrapper::marginalize, src/graph_wrapper.h:17-81 / graph_wrapper_g2o.cpp:398-453)."""

    def __init__(self, path=None, dim=None):
        L = lib()
        _graph_protos(L)
        self.h = C.c_void_p()
        if path is not None:
            _check(L.spg_graph_load_g2o(C.byref(self.h), os.fsencode(path)))
        else:
            _check(L.spg_graph_create(C.byref(self.h), int(dim)))
        self.dim = L.spg_graph_dim(self.h)
        self.P = 3 if self.dim == 3 else 7

    def close(self):
        if getattr(self, "h", None):
            lib().spg_graph_destroy(self.h)
            self.h = None

    def __del__(self):
        self.close()

    def add_vertex(self, vid, pose):
        p = np.ascontiguousarray(pose, dtype=np.float64)
        _check(lib().spg_graph_add_vertex(self.h, int(vid), _p(p)))

    def add_edge(self, a, b, meas, info):
        m = np.ascontiguousarray(meas, dtype=np.float64)
        i = np.ascontiguousarray(np.asarray(info, dtype=np.float64).T)
        _check(lib().spg_graph_add_edge(self.h, int(a), int(b), _p(m), _p(i)))

    def add_factor(self, kind, verts, rows, meas, info, pairs=None):
        """Generic factor (spg_graph_add_factor). info: POSE / MULTI symmetric matrix, GLC the W matrix (rows x d*nv)."""
        v = np.ascontiguousarray(verts, dtype=np.int32)
        m = np.ascontiguousarray(meas, dtype=np.float64).reshape(-1)
        i = np.asarray(info, dtype=np.float64)
        i = np.ascontiguousarray(i.T if kind != 1 else i).reshape(-1)   # column-major for POSE / MULTI, row-major W
        pr = np.ascontiguousarray(pairs, dtype=np.int32) if pairs is not None else None
        _check(lib().spg_graph_add_factor(self.h, int(kind), len(v), _p(v), int(rows), _p(m), _p(i), _p(pr)))

    def set_vertex_pose(self, vid, pose):
        p = np.ascontiguousarray(pose, dtype=np.float64)
        _check(lib().spg_graph_set_vertex_pose(self.h, int(vid), _p(p)))

    def kld(self, ctx, sparse, fixed_id=0):
        """GraphWrapperG2O::kullbackLeibler(other): self = full graph, sparse = sparsified graph -> (kld, terms dict)."""
        v, t = C.c_double(), KldTerms()
        _check(lib().spg_graph_kld(ctx.h, self.h, sparse.h, int(fixed_id), C.byref(v), C.byref(t)))
        return float(v.value), {f: getattr(t, f) for f, _ in KldTerms._fields_}

    def optimize(self, ctx, fixed=(0,), max_iterations=50):
        """GraphWrapperG2O::optimize (g2o Levenberg-Marquardt on the GPU) -> stats dict.

        The linear solve is a dense blocked Cholesky wherever the dense system fits (up to ~122 k free dimensions and
        enough free device memory for two n x n buffers), and block-sparse preconditioned conjugate gradients beyond
        that. stats["solver"] says which ran (SOLVER_DENSE_CHOLESKY / SOLVER_SPARSE_PCG); on the sparse path
        stats["cg_iterations"] sums the CG iterations over all trials and stats["cg_max_rel_residual"] is the worst
        ||r|| / ||b|| at which a trial stopped. The environment variable SPG_OPT_DENSE_MAX_DIMS, read on every call,
        lowers the dense limit (for tests)."""
        f = np.ascontiguousarray(list(fixed), dtype=np.int32)
        st = OptimizeStats()
        _check(lib().spg_graph_optimize(ctx.h, self.h, _p(f), len(f), int(max_iterations), C.byref(st)))
        return {k: getattr(st, k) for k, _ in OptimizeStats._fields_}

    def chi2(self, ctx):
        v = C.c_double()
        _check(lib().spg_graph_chi2(ctx.h, self.h, C.byref(v)))
        return float(v.value)

    def save(self, path):
        """GraphWrapperG2O::write: g2o text with GLC_EDGE / MULTI_EDGE_* factors."""
        _check(lib().spg_graph_save_g2o(self.h, os.fsencode(path)))

    @property
    def num_vertices(self):
        return lib().spg_graph_num_vertices(self.h)

    @property
    def num_edges(self):
        return lib().spg_graph_num_edges(self.h)

    @property
    def max_vertex_id(self):
        return lib().spg_graph_max_vertex_id(self.h)

    def vertex_ids(self):
        ids = np.zeros(self.num_vertices, dtype=np.int32)
        _check(lib().spg_graph_vertex_ids(self.h, _p(ids)))
        return ids

    def vertex_pose(self, vid):
        p = np.zeros(self.P)
        _check(lib().spg_graph_vertex_pose(self.h, int(vid), _p(p)))
        return p

    def marginalize(self, ctx, which, opts, algorithm, allow_failed=False):
        """VertexRemover::remove(which) through the GPU; returns the marginalize stats.
        SPG_ERR_BLANKET_FAILED (6) raises unless allow_failed: the stats then name the first failing entry."""
        w = np.ascontiguousarray(which, dtype=np.int32)
        rc = lib().spg_graph_marginalize(self.h, ctx.h, _p(w), len(w), C.byref(opts), int(algorithm))
        if not (allow_failed and rc == 6):
            _check(rc)
        return self.stats()

    def stats(self):
        s = MarginalizeStats()
        _check(lib().spg_graph_last_stats(self.h, C.byref(s)))
        return {f: getattr(s, f) for f, _ in MarginalizeStats._fields_}

    def edges(self):
        L = lib()
        res = []
        d = EdgeDesc()
        for i in range(self.num_edges):
            _check(L.spg_graph_edge_desc(self.h, i, C.byref(d)))
            ids = np.zeros(d.nv, dtype=np.int32)
            if d.kind == 0:
                meas, info = np.zeros(self.P), np.zeros(self.dim * self.dim)
            elif d.kind == 1:
                meas, info = np.zeros(self.dim * d.nv), np.zeros(d.rows * self.dim * d.nv)
            else:
                meas, info = np.zeros((d.rows // self.dim) * self.P), np.zeros(d.rows * d.rows)
            _check(L.spg_graph_edge_data(self.h, i, _p(ids), _p(meas), _p(info)))
            if d.kind == 0:
                info = info.reshape(self.dim, self.dim).T
            elif d.kind == 1:
                info = info.reshape(d.rows, self.dim * d.nv)
            else:
                info = info.reshape(d.rows, d.rows).T
            rec = {"kind": d.kind, "v": ids, "rows": d.rows, "uid": (d.uid_major, d.uid_minor), "meas": meas, "info": info}
            if d.kind == 2:
                pr = np.zeros(2 * (d.rows // self.dim), dtype=np.int32)
                _check(L.spg_graph_edge_pairs(self.h, i, _p(pr)))
                rec["pairs"] = pr
            res.append(rec)
        return res

    def compute_substitute_edge(self, marginalized, maxid, frm, to):
        """computeSubstituteEdge (src/compute_substitute_edge.cpp:13-96) -> (from, to, meas, info)."""
        m = np.ascontiguousarray(sorted(marginalized), dtype=np.int32)
        f, t = C.c_int32(int(frm)), C.c_int32(int(to))
        meas, info = np.zeros(self.P), np.zeros(self.dim * self.dim)
        _check(lib().spg_compute_substitute_edge(self.h, _p(m), len(m), int(maxid), C.byref(f), C.byref(t), _p(meas), _p(info)))
        return f.value, t.value, meas, info.reshape(self.dim, self.dim).T


def parse_job(line):
    """parseLine (reference src/main.cpp:9-103) -> EvaluateInfo (its g2oname buffer is kept alive on the object)."""
    L = lib()
    L.spg_evaluate_parse_job.argtypes = [C.c_char_p, C.POINTER(EvaluateInfo), C.c_void_p, C.c_int32]
    info = EvaluateInfo()
    buf = C.create_string_buffer(1024)
    _check(L.spg_evaluate_parse_job(line.encode(), C.byref(info), buf, 1024))
    info._buf = buf
    return info


def evaluate(ctx, graph, info, destdir=None, want_graphs=False, cap=100000):
    """evaluate(gw, info) (reference src/evaluate.cpp:32-221) -> dict(samples=[(vertex, value)], result fields...,
    incremental=Graph, baseline=Graph when want_graphs)."""
    L = lib()
    _graph_protos(L)
    L.spg_evaluate.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(EvaluateInfo), C.c_void_p, C.c_void_p, C.c_int32,
                               C.POINTER(EvaluateResult), C.POINTER(C.c_void_p), C.POINTER(C.c_void_p)]
    if destdir is not None:
        info.destdir = os.fsencode(destdir)
    sv, sk = np.zeros(cap, dtype=np.int32), np.zeros(cap, dtype=np.float64)
    res = EvaluateResult()
    inc, base = C.c_void_p(), C.c_void_p()
    rc = L.spg_evaluate(ctx.h, graph.h, C.byref(info), _p(sv), _p(sk), cap, C.byref(res),
                        C.byref(inc) if want_graphs else None, C.byref(base) if want_graphs else None)
    _check(rc)
    out = {f: getattr(res, f) for f, _ in EvaluateResult._fields_}
    n = min(res.n_samples, cap)
    out["samples"] = list(zip(sv[:n].tolist(), sk[:n].tolist()))
    if want_graphs:
        for key, h in (("incremental", inc), ("baseline", base)):
            g = Graph.__new__(Graph)
            g.h = h
            g.dim = L.spg_graph_dim(h)
            g.P = 3 if g.dim == 3 else 7
            out[key] = g
    return out


def decimate_global(last, endvert, sparsity):
    _graph_protos(lib())
    out = np.zeros(max(endvert + 1, 1), dtype=np.int32)
    n = lib().spg_decimate_global(last, endvert, sparsity, _p(out), len(out))
    return out[:n]


def decimate_online(last, endvert, sparsity):
    _graph_protos(lib())
    out = np.zeros(4, dtype=np.int32)
    n = lib().spg_decimate_online(last, endvert, sparsity, _p(out), len(out))
    return out[:n]


def decimate_cluster(last, endvert, sparsity, cluster):
    _graph_protos(lib())
    out = np.zeros(max(endvert + 1, 1), dtype=np.int32)
    n = lib().spg_decimate_cluster(last, endvert, sparsity, cluster, _p(out), len(out))
    return out[:n]


# ---- round-by-round removal (sharding a round over ranks / GPUs) ------------------------------------

def _round_protos(L):
    if getattr(L, "_round_protos_done", False):
        return
    _graph_protos(L)
    L.spg_graph_rounds_begin.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.POINTER(SparsityOptions), C.c_int32]
    L.spg_graph_round_next.argtypes = [C.c_void_p, C.POINTER(RoundIn)]
    L.spg_graph_round_apply.argtypes = [C.c_void_p, C.c_void_p]
    L._round_protos_done = True


def rounds_begin(graph, which, opts, algorithm):
    L = lib()
    _round_protos(L)
    w = np.ascontiguousarray(which, dtype=np.int32)
    _check(L.spg_graph_rounds_begin(graph.h, _p(w), len(w), C.byref(opts), int(algorithm)))


def round_next(graph):
    """Next wavefront round as numpy copies: dict(dim, algorithm, opts, n, records, rec_off, out_off) or None."""
    L = lib()
    _round_protos(L)
    r = RoundIn()
    _check(L.spg_graph_round_next(graph.h, C.byref(r)))
    n = r.n_blankets
    if n == 0:
        return None
    rec_off = np.ctypeslib.as_array(C.cast(r.rec_off, C.POINTER(C.c_int64)), shape=(n + 1,)).copy()
    out_off = np.ctypeslib.as_array(C.cast(r.out_off, C.POINTER(C.c_int64)), shape=(n + 1,)).copy()
    records = np.ctypeslib.as_array(C.cast(r.records, C.POINTER(C.c_uint64)), shape=(int(rec_off[-1]),)).copy()
    return {"dim": r.dim, "algorithm": r.algorithm, "opts": r.opts, "n": n, "records": records, "rec_off": rec_off,
            "out_off": out_off}


def round_apply(graph, out):
    L = lib()
    _round_protos(L)
    out = np.ascontiguousarray(out, dtype=np.uint64)
    _check(L.spg_graph_round_apply(graph.h, _p(out)))
