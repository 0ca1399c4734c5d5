// spg_eval.cu — whole-graph evaluator and optimiser on the GPU (SURVEY.md §8(f) rows 1-2), C ABI in include/spg_capi.h:
//   spg_graph_kld       GraphWrapperG2O::kullbackLeibler   (reference src/graph_wrapper_g2o.cpp:531-548, computeIndices
//                       :472-499, estimateDifference :550-575, kullbackLeiblerDivergence src/utils.cpp:70-97)
//   spg_graph_optimize  GraphWrapperG2O::optimize          (:250-269: g2o Levenberg-Marquardt, 50 iterations, vertex 0 fixed)
//   spg_graph_chi2      GraphWrapperG2O::chi2 / chi2(other) (:501-528)
// The reference solves with CHOLMOD on the sparse system and a dense LDLT for the KLD; here the information matrix is
// assembled dense in HBM (one thread per pose edge, one CTA per GLC factor, fp64 atomics) and factorised with the blocked
// kernels of spg_dense.cuh — GEMM-shaped FP64 work, thousands of dimensions wide. 180 GB of HBM hold graphs of ~100 k
// dimensions this way. Larger KLDs are refused (SPG_ERR_UNSUPPORTED), not approximated; the optimiser assembles larger
// systems block-sparse (the same kernels with another addressing policy) and solves them by PCG (spg_sparse.cuh).
#include <algorithm>
#include <cmath>
#include <cstring>
#include <limits>
#include <memory>
#include <string>
#include <vector>

#include "spg_ctx.h"
#include "spg_dense.cuh"
#include "spg_glc.cuh"
#include "spg_host.h"
#include "spg_sparse.cuh"

namespace {

using spg::Graph;
using spg::GraphEdge;

// ---- flat device view of a graph -----------------------------------------------------------------------------------
struct EdgeRef {
    int32_t kind, nv, rows, pad;
    int64_t vert; // offset into the vertex-index array
    int64_t data; // offset into the payload array (meas then info / W)
    int64_t scratch; // GLC: offset into the scratch array
};

struct DeviceGraph {
    int dim = 0, P = 0, nV = 0;
    std::vector<int> ids;        // ascending
    std::vector<double> poses;   // nV x P (flat poses)
    std::vector<int> verts;      // per edge: local vertex indices
    std::vector<double> data;
    std::vector<EdgeRef> pose_edges, glc_edges, multi_edges;
    int64_t scratch_doubles = 0;
};

void flatten(const Graph &g, DeviceGraph &dg) {
    dg.dim = g.dim;
    dg.P = g.poseWords();
    dg.ids = g.vertexIds();
    dg.nV = (int) dg.ids.size();
    dg.poses.resize((size_t) dg.nV * dg.P);
    std::vector<int> local(g.verts.size(), -1);
    for(int i = 0; i < dg.nV; i++) {
        const int xi = g.indexOf(dg.ids[i]);
        local[xi] = i;
        std::memcpy(&dg.poses[(size_t) i * dg.P], g.verts[xi].pose, sizeof(double) * dg.P);
    }
    for(int ei : g.edgeOrder()) {
        const GraphEdge &e = g.edges[ei];
        EdgeRef r{};
        r.kind = e.kind;
        r.nv = e.nv();
        r.rows = e.rows;
        r.vert = (int64_t) dg.verts.size();
        r.data = (int64_t) dg.data.size();
        for(int q = 0; q < e.nv(); q++) dg.verts.push_back(local[e.vx(q)]);
        if(e.kind == SPG_EDGE_MULTI) // the measurement -> vertex pairs follow the vertex indices
            for(int x : e.pairs) dg.verts.push_back(x);
        dg.data.insert(dg.data.end(), e.payload.begin(), e.payload.end());
        if(e.kind == SPG_EDGE_GLC) {
            const int c = g.dim * e.nv();
            r.scratch = dg.scratch_doubles;
            dg.scratch_doubles += 2 * (int64_t) e.nv() * g.dim * g.dim + (int64_t) e.rows * c + c + e.rows;
            dg.glc_edges.push_back(r);
        } else if(e.kind == SPG_EDGE_MULTI) {
            const int c = g.dim * e.nv();
            r.scratch = dg.scratch_doubles;
            dg.scratch_doubles += 2 * (int64_t) e.rows * c + 2 * (int64_t) e.rows;
            dg.multi_edges.push_back(r);
        } else {
            dg.pose_edges.push_back(r);
        }
    }
}

// ---- device side -------------------------------------------------------------------------------------------------------
template <int D>
__device__ __forceinline__ void pose_from_flat(const double *v, double *p) {
    if constexpr(D == 6) spg::se3_from_flat(v, p);
    else spg::se2_from_flat(v, p);
}

// edge error: SE2 EdgeSE2ISAM::computeError (src/se2_compatibility.h:26-33), SE3 g2o::EdgeSE3 toVectorMQT(Z^-1 Xi^-1 Xj)
template <int D>
__device__ __forceinline__ void edge_error(const double *Z, const double *Xi, const double *Xj, double *e) {
    constexpr int PS = spg::PoseStride<D>::value;
    double T[PS], B[PS];
    if constexpr(D == 6) {
        double A[PS], E[PS];
        spg::se3_inverse(Xi, T);
        spg::se3_compose(T, Xj, B);
        spg::se3_inverse(Z, A);
        spg::se3_compose(A, B, E);
        spg::se3_to_mqt(E, e);
    } else {
        spg::se2_inverse(Xi, T);
        spg::se2_compose(T, Xj, B);
        e[0] = B[0] - Z[0];
        e[1] = B[1] - Z[1];
        e[2] = spg::normalize_theta(B[2] - Z[2]);
    }
}

struct AsmParams {
    const double *poses; // nV x P
    const int32_t *pos;  // per vertex: first row/column in the matrix, -1 = fixed (not a variable)
    const int32_t *verts;
    const double *data;
    const EdgeRef *edges;
    int n_edges;
    double *H;   // n x n column-major (may be NULL: error / gradient only)
    int64_t ldh;
    double *g;   // gradient sum J^T Omega e (may be NULL)
    double *chi2; // sum e^T Omega e (may be NULL)
    double *scratch;
    const int32_t *slots;    // BSR: per factor, the slot of its block pair (a, b) at slot_off[edge] + a + b * nv
    const int64_t *slot_off; // BSR: per factor of the launched kind
};

// Where the D x D block of H at (vertex a of the factor, vertex b of the factor) lives. pr / pc: first row / column of
// the two vertices (pos), ia / ib: their places among the factor's nv vertices.
struct DenseH { // n x n column-major, leading dimension ldh
    struct Blk { int pr, pc; };
    template <int D>
    static __device__ __forceinline__ Blk block(const AsmParams &p, int ei, int nv, int ia, int ib, int pr, int pc) { return {pr, pc}; }
    template <int D>
    static __device__ __forceinline__ double *at(const AsmParams &p, Blk b, int r, int c) { return &p.H[(b.pr + r) + (int64_t) (b.pc + c) * p.ldh]; }
};
struct BsrH { // one D x D column-major block per slot (spg_sparse.cuh)
    using Blk = double *;
    template <int D>
    static __device__ __forceinline__ Blk block(const AsmParams &p, int ei, int nv, int ia, int ib, int pr, int pc) {
        return p.H + (int64_t) p.slots[p.slot_off[ei] + ia + ib * nv] * (D * D);
    }
    template <int D>
    static __device__ __forceinline__ double *at(const AsmParams &p, Blk b, int r, int c) { return b + r + c * D; }
};

// one thread per pose edge: H += J^T Omega J, g += J^T Omega e, chi2 += e^T Omega e
template <int D, class A>
__global__ void __launch_bounds__(64) assemble_pose_edges_kernel(const AsmParams p) {
    constexpr int PS = spg::PoseStride<D>::value, PW = (D == 6) ? 7 : 3;
    double chi = 0.0;
    for(int ei = blockIdx.x * blockDim.x + threadIdx.x; ei < p.n_edges; ei += gridDim.x * blockDim.x) {
        const EdgeRef er = p.edges[ei];
        const int va = p.verts[er.vert], vb = p.verts[er.vert + 1];
        const double *pl = p.data + er.data;
        const double *Om = pl + PW; // D x D column-major
        double Z[PS], Xi[PS], Xj[PS], J[2 * D * D], e[D], Oe[D];
        pose_from_flat<D>(pl, Z);
        pose_from_flat<D>(p.poses + (size_t) va * PW, Xi);
        pose_from_flat<D>(p.poses + (size_t) vb * PW, Xj);
        edge_error<D>(Z, Xi, Xj, e);
        for(int r = 0; r < D; r++) {
            double s = 0;
            for(int c = 0; c < D; c++) s += Om[r + c * D] * e[c];
            Oe[r] = s;
        }
        for(int r = 0; r < D; r++) chi += e[r] * Oe[r];
        if(!p.H && !p.g) continue;
        spg::edge_jacobians<D>(Z, Xi, Xj, J); // J[0 .. D*D): d e / d xi, J[D*D ..): d e / d xj, column-major D x D
        const int pa = p.pos[va], pb = p.pos[vb];
        if(p.g) {
            for(int side = 0; side < 2; side++) {
                const int pv = side ? pb : pa;
                if(pv < 0) continue;
                const double *Js = J + side * D * D;
                for(int c = 0; c < D; c++) {
                    double s = 0;
                    for(int r = 0; r < D; r++) s += Js[r + c * D] * Oe[r];
                    atomicAdd(&p.g[pv + c], s);
                }
            }
        }
        if(p.H) {
            double M[2 * D * D]; // Omega * J
            for(int side = 0; side < 2; side++)
                for(int c = 0; c < D; c++)
                    for(int r = 0; r < D; r++) {
                        double s = 0;
                        for(int q = 0; q < D; q++) s += Om[r + q * D] * J[side * D * D + q + c * D];
                        M[side * D * D + r + c * D] = s;
                    }
            for(int sa = 0; sa < 2; sa++) {
                const int pr = sa ? pb : pa;
                if(pr < 0) continue;
                for(int sb = 0; sb < 2; sb++) {
                    const int pc = sb ? pb : pa;
                    if(pc < 0) continue;
                    const typename A::Blk blk = A::template block<D>(p, ei, 2, sa, sb, pr, pc);
                    for(int c = 0; c < D; c++)
                        for(int r = 0; r < D; r++) {
                            double s = 0;
                            for(int q = 0; q < D; q++) s += J[sa * D * D + q + r * D] * M[sb * D * D + q + c * D];
                            atomicAdd(A::template at<D>(p, blk, r, c), s);
                        }
                }
            }
        }
    }
    if(p.chi2) {
        for(int o = 16; o > 0; o >>= 1) chi += __shfl_down_sync(0xffffffffu, chi, o);
        if((threadIdx.x & 31) == 0) atomicAdd(p.chi2, chi);
    }
}

// one CTA per GLC factor: J = W * J_reparam (GLCEdge::linearizeOplus, src/glc_edge.cpp:40-49), error = W * r
// (computeError :28-32), Omega = I
template <int D, class A>
__global__ void __launch_bounds__(64) assemble_glc_edges_kernel(const AsmParams p) {
    constexpr int PS = spg::PoseStride<D>::value, PW = (D == 6) ? 7 : 3, NT = 64;
    const int tid = threadIdx.x;
    for(int ei = blockIdx.x; ei < p.n_edges; ei += gridDim.x) {
        const EdgeRef er = p.edges[ei];
        const int nv = er.nv, r = er.rows, c = D * nv;
        const int32_t *vi = p.verts + er.vert;
        const double *meas = p.data + er.data;
        const double *W = meas + c; // r x c row-major
        double *JA = p.scratch + er.scratch, *JB = JA + nv * D * D, *Jf = JB + nv * D * D; // Jf: r x c column-major
        double *rv = Jf + (size_t) r * c, *err = rv + c;
        __syncthreads();
        for(int i = tid; i < nv; i += NT) {
            double x0[PS], xi[PS], Z[PS], e[D];
            pose_from_flat<D>(p.poses + (size_t) vi[0] * PW, x0);
            pose_from_flat<D>(p.poses + (size_t) vi[i] * PW, xi);
            spg::glc_reparam_blocks<D>(i, meas, x0, xi, JA + i * D * D, JB + i * D * D);
            spg::glc_error_to_pose<D>(meas + i * D, Z);
            if(i == 0) {
                double I0[PS];
                spg::pose_identity<D>(I0);
                edge_error<D>(Z, I0, x0, e);
            } else {
                edge_error<D>(Z, x0, xi, e);
            }
            for(int q = 0; q < D; q++) rv[i * D + q] = e[q];
        }
        __syncthreads();
        for(int t = tid; t < r * c; t += NT) {
            const int row = t % r, col = t / r, bi = col / D, j = col % D;
            double s = 0;
            if(bi == 0) {
                for(int i = 0; i < nv; i++)
                    for(int q = 0; q < D; q++) s += W[(size_t) row * c + i * D + q] * JA[i * D * D + q + j * D];
            } else {
                for(int q = 0; q < D; q++) s += W[(size_t) row * c + bi * D + q] * JB[bi * D * D + q + j * D];
            }
            Jf[row + (size_t) col * r] = s;
        }
        for(int row = tid; row < r; row += NT) {
            double s = 0;
            for(int q = 0; q < c; q++) s += W[(size_t) row * c + q] * rv[q];
            err[row] = s;
        }
        __syncthreads();
        if(p.chi2 && tid == 0) {
            double s = 0;
            for(int row = 0; row < r; row++) s += err[row] * err[row];
            atomicAdd(p.chi2, s);
        }
        if(p.g)
            for(int a = tid; a < c; a += NT) {
                const int pv = p.pos[vi[a / D]];
                if(pv < 0) continue;
                double s = 0;
                for(int row = 0; row < r; row++) s += Jf[row + (size_t) a * r] * err[row];
                atomicAdd(&p.g[pv + a % D], s);
            }
        if(p.H)
            for(int t = tid; t < c * c; t += NT) {
                const int a = t % c, b = t / c;
                const int pa = p.pos[vi[a / D]], pb = p.pos[vi[b / D]];
                if(pa < 0 || pb < 0) continue;
                double s = 0;
                for(int row = 0; row < r; row++) s += Jf[row + (size_t) a * r] * Jf[row + (size_t) b * r];
                atomicAdd(A::template at<D>(p, A::template block<D>(p, ei, nv, a / D, b / D, pa, pb), a % D, b % D), s);
            }
    }
}

// one CTA per MultiEdgeCorrelated (multi_edge_correlated.hpp:64-140): stacked pose errors and Jacobians, full Omega
template <int D, class A>
__global__ void __launch_bounds__(64) assemble_multi_edges_kernel(const AsmParams p) {
    constexpr int PS = spg::PoseStride<D>::value, PW = (D == 6) ? 7 : 3, NT = 64;
    const int tid = threadIdx.x;
    for(int ei = blockIdx.x; ei < p.n_edges; ei += gridDim.x) {
        const EdgeRef er = p.edges[ei];
        const int nv = er.nv, rows = er.rows, nm = rows / D, c = D * nv;
        const int32_t *vi = p.verts + er.vert, *pr = vi + nv;
        const double *meas = p.data + er.data;
        const double *Om = meas + (size_t) nm * PW; // rows x rows column-major
        double *Jf = p.scratch + er.scratch, *M = Jf + (size_t) rows * c, *err = M + (size_t) rows * c, *Oe = err + rows;
        __syncthreads();
        for(int t = tid; t < rows * c; t += NT) Jf[t] = 0.0;
        __syncthreads();
        for(int q = tid; q < nm; q += NT) {
            double Z[PS], Xa[PS], Xb[PS], J[2 * D * D], e[D];
            const int a = pr[2 * q], b = pr[2 * q + 1];
            pose_from_flat<D>(meas + (size_t) q * PW, Z);
            pose_from_flat<D>(p.poses + (size_t) vi[a] * PW, Xa);
            pose_from_flat<D>(p.poses + (size_t) vi[b] * PW, Xb);
            edge_error<D>(Z, Xa, Xb, e);
            spg::edge_jacobians<D>(Z, Xa, Xb, J);
            for(int r = 0; r < D; r++) {
                err[q * D + r] = e[r];
                for(int l = 0; l < D; l++) {
                    Jf[(q * D + r) + (size_t) (a * D + l) * rows] = J[r + l * D];
                    Jf[(q * D + r) + (size_t) (b * D + l) * rows] = J[D * D + r + l * D];
                }
            }
        }
        __syncthreads();
        for(int row = tid; row < rows; row += NT) {
            double s = 0;
            for(int q = 0; q < rows; q++) s += Om[row + (size_t) q * rows] * err[q];
            Oe[row] = s;
        }
        if(p.H)
            for(int t = tid; t < rows * c; t += NT) {
                const int row = t % rows, col = t / rows;
                double s = 0;
                for(int q = 0; q < rows; q++) s += Om[row + (size_t) q * rows] * Jf[q + (size_t) col * rows];
                M[t] = s;
            }
        __syncthreads();
        if(p.chi2 && tid == 0) {
            double s = 0;
            for(int row = 0; row < rows; row++) s += err[row] * Oe[row];
            atomicAdd(p.chi2, s);
        }
        if(p.g)
            for(int a = tid; a < c; a += NT) {
                const int pv = p.pos[vi[a / D]];
                if(pv < 0) continue;
                double s = 0;
                for(int row = 0; row < rows; row++) s += Jf[row + (size_t) a * rows] * Oe[row];
                atomicAdd(&p.g[pv + a % D], s);
            }
        if(p.H)
            for(int t = tid; t < c * c; t += NT) {
                const int a = t % c, b = t / c;
                const int pa = p.pos[vi[a / D]], pb = p.pos[vi[b / D]];
                if(pa < 0 || pb < 0) continue;
                double s = 0;
                for(int row = 0; row < rows; row++) s += Jf[row + (size_t) a * rows] * M[row + (size_t) b * rows];
                atomicAdd(A::template at<D>(p, A::template block<D>(p, ei, nv, a / D, b / D, pa, pb), a % D, b % D), s);
            }
    }
}

__global__ void add_diag_kernel(double *A, int64_t lda, int n, double lambda) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if(i < n) A[i + (int64_t) i * lda] += lambda;
}
__global__ void max_diag_kernel(const double *A, int64_t lda, int n, double *out) { // single CTA
    double m = 0;
    for(int i = threadIdx.x; i < n; i += blockDim.x) m = fmax(m, A[i + (int64_t) i * lda]);
    for(int o = 16; o > 0; o >>= 1) m = fmax(m, __shfl_down_sync(0xffffffffu, m, o));
    __shared__ double part[32];
    if((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = m;
    __syncthreads();
    if(threadIdx.x == 0) {
        for(int w = 1; w < (int) (blockDim.x >> 5); w++) m = fmax(m, part[w]);
        *out = m;
    }
}
// x_j <- L_jj^-T x_j for one nb x nb diagonal block (single thread: nb <= 64)
__global__ void trsv_t_block_kernel(const double *L, int64_t ldl, int nb, double *x) {
    if(threadIdx.x != 0 || blockIdx.x != 0) return;
    for(int i = nb - 1; i >= 0; i--) {
        double s = x[i];
        for(int p = i + 1; p < nb; p++) s -= L[p + (int64_t) i * ldl] * x[p];
        x[i] = s / L[i + (int64_t) i * ldl];
    }
}
// y[c] -= sum_i L[j0 + i, c] * x[i]  for c < ncols (the block row j0 .. j0+nb of a lower factor, transposed)
__global__ void gemv_t_sub_kernel(const double *L, int64_t ldl, int nb, int ncols, const double *x, double *y) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if(c >= ncols) return;
    const double *col = L + (int64_t) c * ldl;
    double s = 0;
    for(int i = 0; i < nb; i++) s = fma(col[i], x[i], s);
    y[c] -= s;
}

// ---- host-side drivers of the blocked kernels (all on `st`) ---------------------------------------------------------
bool g_dense_configured = false;
cudaError_t configure_dense() {
    if(g_dense_configured) return cudaSuccess;
    cudaError_t e = cudaFuncSetAttribute(spg::trsm_right_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, spg::DENSE_TRSM_SMEM);
    if(e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(spg::trsm_left_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, spg::DENSE_TRSM_SMEM);
    if(e == cudaSuccess) g_dense_configured = true;
    return e;
}

// blocked right-looking Cholesky of the first `ncols` columns of the n x n matrix A (lower triangle). ncols == n:
// A = L L^T; ncols < n: the trailing block becomes the Schur complement A22 - A21 A11^-1 A12 (lower triangle).
void cholesky_partial(spg_ctx *ctx, double *A, int64_t lda, int n, int ncols, double *logdet, int *flag) {
    cudaStream_t st = ctx->stream;
    for(int j0 = 0; j0 < ncols; j0 += spg::DNB) {
        const int nb = std::min(spg::DNB, ncols - j0);
        double *Ajj = A + j0 + (int64_t) j0 * lda;
        spg::potrf_block_kernel<<<1, 256, 0, st>>>(Ajj, lda, nb, logdet, flag);
        const int rows = n - j0 - nb;
        if(rows > 0) {
            double *P = Ajj + nb;
            spg::trsm_right_kernel<<<(rows + 63) / 64, 64, spg::DENSE_TRSM_SMEM, st>>>(Ajj, lda, nb, P, lda, rows);
            double *T = A + (j0 + nb) + (int64_t) (j0 + nb) * lda;
            dim3 grid((rows + 63) / 64, (rows + 63) / 64);
            spg::dgemm_sub_kernel<true><<<grid, 256, 0, st>>>(rows, rows, nb, P, lda, P, lda, T, lda, 1);
        }
        ctx->launches += rows > 0 ? 3 : 1;
    }
}

// forward substitution L Z = B with a lower factor L (n x n) and B (n x cols), in place
void forward_solve(spg_ctx *ctx, const double *L, int64_t ldl, int n, double *B, int64_t ldb, int cols) {
    cudaStream_t st = ctx->stream;
    for(int j0 = 0; j0 < n; j0 += spg::DNB) {
        const int nb = std::min(spg::DNB, n - j0);
        const double *Ljj = L + j0 + (int64_t) j0 * ldl;
        double *Bj = B + j0;
        spg::trsm_left_kernel<<<(cols + 63) / 64, 64, spg::DENSE_TRSM_SMEM, st>>>(Ljj, ldl, nb, Bj, ldb, cols);
        const int rows = n - j0 - nb;
        if(rows > 0) {
            dim3 grid((rows + 63) / 64, (cols + 63) / 64);
            spg::dgemm_sub_kernel<false><<<grid, 256, 0, st>>>(rows, cols, nb, Ljj + nb, ldl, Bj, ldb, Bj + nb, ldb, 0);
        }
        ctx->launches += rows > 0 ? 2 : 1;
    }
}

// backward substitution L^T x = y for one right-hand side, in place
void backward_solve_vec(spg_ctx *ctx, const double *L, int64_t ldl, int n, double *x) {
    cudaStream_t st = ctx->stream;
    const int nblk = (n + spg::DNB - 1) / spg::DNB;
    for(int b = nblk - 1; b >= 0; b--) {
        const int j0 = b * spg::DNB, nb = std::min(spg::DNB, n - j0);
        trsv_t_block_kernel<<<1, 32, 0, st>>>(L + j0 + (int64_t) j0 * ldl, ldl, nb, x + j0);
        if(j0 > 0) gemv_t_sub_kernel<<<(j0 + 127) / 128, 128, 0, st>>>(L + j0, ldl, nb, j0, x + j0, x);
        ctx->launches += j0 > 0 ? 2 : 1;
    }
}

// Block pattern of H over the free vertices for the sparse path (spg_sparse.cuh): block rows in layout() order, a block
// for every ordered pair of free vertices of a factor (pose edges 2 x 2; GLC and MULTI nv x nv, since their Omega
// couples every row) and every diagonal block, both triangles stored.
struct Bsr {
    int nb = 0;
    int64_t nnzb = 0;
    std::vector<int32_t> rowptr, col, diag; // diag: slot of each row's diagonal block
    std::vector<int32_t> slots;             // per factor (pose, GLC, then MULTI edges): nv x nv, -1 where a vertex is fixed
    std::vector<int64_t> slot_off;          // per factor: offset of its table in slots
};

template <class F>
void for_each_factor(const DeviceGraph &dg, F f) {
    for(const auto *list : {&dg.pose_edges, &dg.glc_edges, &dg.multi_edges})
        for(const EdgeRef &e : *list) f(e);
}

spg_status build_bsr(const DeviceGraph &dg, const std::vector<int32_t> &pos, int n, Bsr &b) {
    const int D = dg.dim;
    b.nb = n / D;
    std::vector<int64_t> start((size_t) b.nb + 1, 0);
    std::vector<int32_t> rows;
    auto free_rows = [&](const EdgeRef &e) {
        rows.clear();
        for(int q = 0; q < e.nv; q++) {
            const int pv = pos[dg.verts[e.vert + q]];
            if(pv >= 0) rows.push_back(pv / D);
        }
    };
    for(int i = 0; i < b.nb; i++) start[i + 1] = 1;
    for_each_factor(dg, [&](const EdgeRef &e) {
        free_rows(e);
        for(int r : rows) start[r + 1] += (int64_t) rows.size();
    });
    for(int i = 0; i < b.nb; i++) start[i + 1] += start[i];
    std::vector<int32_t> cols((size_t) start[b.nb]);
    std::vector<int64_t> fill(start.begin(), start.end() - 1);
    for(int i = 0; i < b.nb; i++) cols[fill[i]++] = i;
    for_each_factor(dg, [&](const EdgeRef &e) {
        free_rows(e);
        for(int r : rows)
            for(int c : rows) cols[fill[r]++] = c;
    });
    b.rowptr.assign((size_t) b.nb + 1, 0);
    b.col.clear();
    for(int i = 0; i < b.nb; i++) {
        auto lo = cols.begin() + start[i], hi = cols.begin() + start[i + 1];
        std::sort(lo, hi);
        b.col.insert(b.col.end(), lo, std::unique(lo, hi));
        if(b.col.size() > (size_t) std::numeric_limits<int32_t>::max()) {
            spg_set_err("spg_graph_optimize: block-sparse system has more than 2^31 blocks");
            return SPG_ERR_UNSUPPORTED;
        }
        b.rowptr[i + 1] = (int32_t) b.col.size();
    }
    b.nnzb = (int64_t) b.col.size();
    auto slot_of = [&](int r, int c) {
        const auto lo = b.col.begin() + b.rowptr[r], hi = b.col.begin() + b.rowptr[r + 1];
        return (int32_t) (std::lower_bound(lo, hi, c) - b.col.begin());
    };
    b.diag.resize((size_t) b.nb);
    for(int i = 0; i < b.nb; i++) b.diag[i] = slot_of(i, i);
    b.slots.clear();
    b.slot_off.clear();
    for_each_factor(dg, [&](const EdgeRef &e) {
        b.slot_off.push_back((int64_t) b.slots.size());
        for(int ib = 0; ib < e.nv; ib++)
            for(int ia = 0; ia < e.nv; ia++) {
                const int pa = pos[dg.verts[e.vert + ia]], pb = pos[dg.verts[e.vert + ib]];
                b.slots.push_back(pa >= 0 && pb >= 0 ? slot_of(pa / D, pb / D) : -1);
            }
    });
    return SPG_OK;
}

struct DevArrays {
    DevBuf poses, pos, verts, data, pedges, gedges, medges, scratch, slots, slot_off;
};

// bsr: the slot tables of the sparse path (NULL: dense H)
spg_status upload(spg_ctx *ctx, const DeviceGraph &dg, const std::vector<int32_t> &pos, DevArrays &d, const Bsr *bsr = nullptr) {
    cudaStream_t st = ctx->stream;
    SPG_CUDA(d.poses.reserve(dg.poses.size() * 8 + 8));
    SPG_CUDA(d.pos.reserve(pos.size() * 4 + 8));
    SPG_CUDA(d.verts.reserve(dg.verts.size() * 4 + 8));
    SPG_CUDA(d.data.reserve(dg.data.size() * 8 + 8));
    SPG_CUDA(d.pedges.reserve(dg.pose_edges.size() * sizeof(EdgeRef) + 8));
    SPG_CUDA(d.gedges.reserve(dg.glc_edges.size() * sizeof(EdgeRef) + 8));
    SPG_CUDA(d.medges.reserve(dg.multi_edges.size() * sizeof(EdgeRef) + 8));
    SPG_CUDA(d.scratch.reserve((size_t) dg.scratch_doubles * 8 + 8));
    SPG_CUDA(cudaMemcpyAsync(d.poses.p, dg.poses.data(), dg.poses.size() * 8, cudaMemcpyHostToDevice, st));
    SPG_CUDA(cudaMemcpyAsync(d.pos.p, pos.data(), pos.size() * 4, cudaMemcpyHostToDevice, st));
    SPG_CUDA(cudaMemcpyAsync(d.verts.p, dg.verts.data(), dg.verts.size() * 4, cudaMemcpyHostToDevice, st));
    SPG_CUDA(cudaMemcpyAsync(d.data.p, dg.data.data(), dg.data.size() * 8, cudaMemcpyHostToDevice, st));
    if(!dg.pose_edges.empty())
        SPG_CUDA(cudaMemcpyAsync(d.pedges.p, dg.pose_edges.data(), dg.pose_edges.size() * sizeof(EdgeRef), cudaMemcpyHostToDevice, st));
    if(!dg.glc_edges.empty())
        SPG_CUDA(cudaMemcpyAsync(d.gedges.p, dg.glc_edges.data(), dg.glc_edges.size() * sizeof(EdgeRef), cudaMemcpyHostToDevice, st));
    if(!dg.multi_edges.empty())
        SPG_CUDA(cudaMemcpyAsync(d.medges.p, dg.multi_edges.data(), dg.multi_edges.size() * sizeof(EdgeRef), cudaMemcpyHostToDevice, st));
    if(bsr) {
        SPG_CUDA(d.slots.reserve(bsr->slots.size() * 4 + 8));
        SPG_CUDA(d.slot_off.reserve(bsr->slot_off.size() * 8 + 8));
        SPG_CUDA(cudaMemcpyAsync(d.slots.p, bsr->slots.data(), bsr->slots.size() * 4, cudaMemcpyHostToDevice, st));
        SPG_CUDA(cudaMemcpyAsync(d.slot_off.p, bsr->slot_off.data(), bsr->slot_off.size() * 8, cudaMemcpyHostToDevice, st));
    }
    return SPG_OK;
}
void release(DevArrays &d) {
    for(DevBuf *b : {&d.poses, &d.pos, &d.verts, &d.data, &d.pedges, &d.gedges, &d.medges, &d.scratch, &d.slots, &d.slot_off}) b->release();
}

// H (zeroed here when given), g (n, zeroed), chi2 (1, zeroed) of the graph at the uploaded poses. H is the n x n dense
// matrix of leading dimension ldh, or with bsr_blocks > 0 the values of that many BSR blocks (slot tables uploaded).
spg_status assemble(spg_ctx *ctx, const DeviceGraph &dg, DevArrays &d, int n, double *H, int64_t ldh, double *g, double *chi2,
                    int64_t bsr_blocks = 0) {
    cudaStream_t st = ctx->stream;
    const bool bsr = bsr_blocks > 0;
    if(H) SPG_CUDA(cudaMemsetAsync(H, 0, bsr ? (size_t) bsr_blocks * dg.dim * dg.dim * 8 : (size_t) ldh * n * 8, st));
    if(g) SPG_CUDA(cudaMemsetAsync(g, 0, (size_t) n * 8, st));
    if(chi2) SPG_CUDA(cudaMemsetAsync(chi2, 0, 8, st));
    AsmParams p{};
    p.poses = static_cast<const double *>(d.poses.p);
    p.pos = static_cast<const int32_t *>(d.pos.p);
    p.verts = static_cast<const int32_t *>(d.verts.p);
    p.data = static_cast<const double *>(d.data.p);
    p.H = H;
    p.ldh = ldh;
    p.g = g;
    p.chi2 = chi2;
    p.scratch = static_cast<double *>(d.scratch.p);
    p.slots = static_cast<const int32_t *>(d.slots.p);
    const int64_t *slot_off = static_cast<const int64_t *>(d.slot_off.p);
#define SPG_ASM_LAUNCH(kernel, blocks)                                       \
    do {                                                                     \
        if(bsr) {                                                            \
            if(dg.dim == 6) kernel<6, BsrH><<<blocks, 64, 0, st>>>(p);       \
            else kernel<3, BsrH><<<blocks, 64, 0, st>>>(p);                  \
        } else {                                                             \
            if(dg.dim == 6) kernel<6, DenseH><<<blocks, 64, 0, st>>>(p);     \
            else kernel<3, DenseH><<<blocks, 64, 0, st>>>(p);                \
        }                                                                    \
        ctx->launches++;                                                     \
    } while(0)
    if(!dg.pose_edges.empty()) {
        p.edges = static_cast<const EdgeRef *>(d.pedges.p);
        p.n_edges = (int) dg.pose_edges.size();
        p.slot_off = slot_off;
        const int blocks = std::min<int>((p.n_edges + 63) / 64, ctx->sm_count * 16);
        SPG_ASM_LAUNCH(assemble_pose_edges_kernel, blocks);
    }
    if(!dg.glc_edges.empty()) {
        p.edges = static_cast<const EdgeRef *>(d.gedges.p);
        p.n_edges = (int) dg.glc_edges.size();
        p.slot_off = slot_off ? slot_off + dg.pose_edges.size() : nullptr;
        const int blocks = std::min<int>(p.n_edges, ctx->sm_count * 16);
        SPG_ASM_LAUNCH(assemble_glc_edges_kernel, blocks);
    }
    if(!dg.multi_edges.empty()) {
        p.edges = static_cast<const EdgeRef *>(d.medges.p);
        p.n_edges = (int) dg.multi_edges.size();
        p.slot_off = slot_off ? slot_off + dg.pose_edges.size() + dg.glc_edges.size() : nullptr;
        const int blocks = std::min<int>(p.n_edges, ctx->sm_count * 16);
        SPG_ASM_LAUNCH(assemble_multi_edges_kernel, blocks);
    }
#undef SPG_ASM_LAUNCH
    SPG_CUDA(cudaGetLastError());
    return SPG_OK;
}

// vertex -> first matrix row; fixed vertices get -1. With `keep`: the marginalised variables first (*n_first of them),
// then the kept ones, each in ascending id; without: all variables in ascending id.
int layout(const DeviceGraph &dg, const std::vector<char> &fixed, const std::vector<char> *keep, std::vector<int32_t> &pos, int *n_first) {
    pos.assign((size_t) dg.nV, -1);
    int k = 0;
    if(keep) {
        for(int i = 0; i < dg.nV; i++)
            if(!fixed[i] && !(*keep)[i]) { pos[i] = k; k += dg.dim; }
    }
    if(n_first) *n_first = k;
    for(int i = 0; i < dg.nV; i++)
        if(!fixed[i] && (!keep || (*keep)[i])) { pos[i] = k; k += dg.dim; }
    return k;
}

// fromVectorMQT / SE2 update of a flat pose (VertexSE3::oplusImpl: X <- X * fromVectorMQT(d); VertexSE2: Euclidean)
void oplus_flat(int dim, double *pose, const double *d) {
    if(dim == 3) {
        pose[0] += d[0];
        pose[1] += d[1];
        double th = pose[2] + d[2];
        while(th > M_PI) th -= 2 * M_PI;
        while(th < -M_PI) th += 2 * M_PI;
        pose[2] = th;
        return;
    }
    double w = 1.0 - (d[3] * d[3] + d[4] * d[4] + d[5] * d[5]);
    double q[7] = {d[0], d[1], d[2], 0, 0, 0, 1};
    if(w >= 0) { // g2o::internal::fromVectorMQT: identity rotation when the vector part is longer than 1
        q[3] = d[3]; q[4] = d[4]; q[5] = d[5]; q[6] = std::sqrt(w);
    }
    double out[7];
    spg::poseCompose(6, pose, q, out);
    std::memcpy(pose, out, sizeof(out));
}

// ---- spg_graph_optimize: one Levenberg-Marquardt driver over two ways of storing and solving the system ----------------
// The steps that depend on the storage of H. g (n doubles) and sc ([0] chi2, [1] max diagonal) belong to the driver.
struct LinearSystem {
    int64_t cg_iterations = 0;
    double cg_max_rel_residual = 0;
    virtual ~LinearSystem() = default;
    // H, g and chi2 at the uploaded poses
    virtual spg_status build(double *g, double *chi2) = 0;
    virtual spg_status max_diag(double *out) = 0;
    // (H + lambda I) x = -g into hx; *ok = false when H + lambda I is not positive definite
    virtual spg_status solve(double lambda, const double *g, const std::vector<double> &hg, std::vector<double> &hx, bool *ok) = 0;
};

// H dense in HBM, blocked Cholesky + forward / backward substitution (spg_dense.cuh)
struct DenseSystem : LinearSystem {
    spg_ctx *ctx;
    const DeviceGraph &dg;
    DevArrays &arr;
    const int n;
    DevBuf dH, dwork, dx, dflag; // H, H + lambda I and its factor, x, Cholesky flag
    DenseSystem(spg_ctx *c, const DeviceGraph &d, DevArrays &a, int n_) : ctx(c), dg(d), arr(a), n(n_) {}
    ~DenseSystem() override {
        for(DevBuf *b : {&dH, &dwork, &dx, &dflag}) b->release();
    }
    cudaError_t reserve() {
        const size_t nn = (size_t) std::max(n, 1);
        cudaError_t e = dH.reserve(nn * nn * 8);
        if(e == cudaSuccess) e = dx.reserve(nn * 8);
        if(e == cudaSuccess) e = dflag.reserve(8);
        if(e == cudaSuccess) e = dwork.reserve(nn * nn * 8);
        return e;
    }
    spg_status build(double *g, double *chi2) override {
        return assemble(ctx, dg, arr, n, static_cast<double *>(dH.p), n, g, chi2);
    }
    spg_status max_diag(double *out) override {
        max_diag_kernel<<<1, 1024, 0, ctx->stream>>>(static_cast<double *>(dH.p), n, n, out);
        return SPG_OK;
    }
    spg_status solve(double lambda, const double *, const std::vector<double> &hg, std::vector<double> &hx, bool *ok) override {
        cudaStream_t st = ctx->stream;
        double *Wk = static_cast<double *>(dwork.p), *x = static_cast<double *>(dx.p);
        int *flag = static_cast<int *>(dflag.p);
        SPG_CUDA(cudaMemcpyAsync(Wk, dH.p, (size_t) n * n * 8, cudaMemcpyDeviceToDevice, st));
        add_diag_kernel<<<(n + 255) / 256, 256, 0, st>>>(Wk, n, n, lambda);
        SPG_CUDA(cudaMemsetAsync(flag, 0, 4, st));
        cholesky_partial(ctx, Wk, n, n, n, nullptr, flag);
        for(int q = 0; q < n; q++) hx[q] = -hg[q];
        SPG_CUDA(cudaMemcpyAsync(x, hx.data(), (size_t) n * 8, cudaMemcpyHostToDevice, st));
        forward_solve(ctx, Wk, n, n, x, n, 1);
        backward_solve_vec(ctx, Wk, n, n, x);
        int hflag = 0;
        SPG_CUDA(cudaMemcpyAsync(hx.data(), x, (size_t) n * 8, cudaMemcpyDeviceToHost, st));
        SPG_CUDA(cudaMemcpyAsync(&hflag, flag, 4, cudaMemcpyDeviceToHost, st));
        SPG_CUDA(cudaStreamSynchronize(st));
        *ok = hflag == 0;
        return SPG_OK;
    }
};

// H block-sparse (BSR, both triangles), block-Jacobi PCG (spg_sparse.cuh)
struct SparseSystem : LinearSystem {
    spg_ctx *ctx;
    const DeviceGraph &dg;
    DevArrays &arr;
    const Bsr &bsr;
    const int n, nb, grid_spmv, grid_rows;
    DevBuf dvals, drowptr, dcol, ddiag, dminv, dx, dr, dz, dp0, dp1, dq, dpart, dstate;
    SparseSystem(spg_ctx *c, const DeviceGraph &d, DevArrays &a, const Bsr &b, int n_)
        : ctx(c), dg(d), arr(a), bsr(b), n(n_), nb(b.nb),
          grid_spmv(std::max(1, std::min((b.nb + 7) / 8, c->sm_count * spg::PCG_CTAS_PER_SM))),
          grid_rows(std::max(1, std::min((b.nb + 255) / 256, c->sm_count * spg::PCG_CTAS_PER_SM))) {}
    ~SparseSystem() override {
        for(DevBuf *b : {&dvals, &drowptr, &dcol, &ddiag, &dminv, &dx, &dr, &dz, &dp0, &dp1, &dq, &dpart, &dstate}) b->release();
    }
    spg_status reserve() {
        cudaStream_t st = ctx->stream;
        const int D = dg.dim;
        const size_t vec = (size_t) n * 8 + 8, part = (size_t) 3 * ctx->sm_count * spg::PCG_CTAS_PER_SM * 8;
        SPG_CUDA(dvals.reserve((size_t) bsr.nnzb * D * D * 8 + 8));
        SPG_CUDA(drowptr.reserve(bsr.rowptr.size() * 4 + 8));
        SPG_CUDA(dcol.reserve(bsr.col.size() * 4 + 8));
        SPG_CUDA(ddiag.reserve(bsr.diag.size() * 4 + 8));
        SPG_CUDA(dminv.reserve((size_t) nb * D * D * 8 + 8));
        for(DevBuf *b : {&dx, &dr, &dz, &dp0, &dp1, &dq}) SPG_CUDA(b->reserve(vec));
        SPG_CUDA(dpart.reserve(part));
        SPG_CUDA(dstate.reserve(sizeof(spg::PcgState)));
        SPG_CUDA(cudaMemcpyAsync(drowptr.p, bsr.rowptr.data(), bsr.rowptr.size() * 4, cudaMemcpyHostToDevice, st));
        SPG_CUDA(cudaMemcpyAsync(dcol.p, bsr.col.data(), bsr.col.size() * 4, cudaMemcpyHostToDevice, st));
        SPG_CUDA(cudaMemcpyAsync(ddiag.p, bsr.diag.data(), bsr.diag.size() * 4, cudaMemcpyHostToDevice, st));
        return SPG_OK;
    }
    spg_status build(double *g, double *chi2) override {
        return assemble(ctx, dg, arr, n, static_cast<double *>(dvals.p), 0, g, chi2, std::max<int64_t>(bsr.nnzb, 1));
    }
    spg_status max_diag(double *out) override {
        const double *v = static_cast<const double *>(dvals.p);
        const int32_t *dd = static_cast<const int32_t *>(ddiag.p);
        if(dg.dim == 6) spg::bsr_max_diag_kernel<6><<<1, 1024, 0, ctx->stream>>>(v, dd, nb, out);
        else spg::bsr_max_diag_kernel<3><<<1, 1024, 0, ctx->stream>>>(v, dd, nb, out);
        return SPG_OK;
    }
    spg_status solve(double lambda, const double *g, const std::vector<double> &, std::vector<double> &hx, bool *ok) override {
        return dg.dim == 6 ? pcg<6>(lambda, g, hx, ok) : pcg<3>(lambda, g, hx, ok);
    }
    template <int D>
    spg_status pcg(double lambda, const double *g, std::vector<double> &hx, bool *ok) {
        cudaStream_t st = ctx->stream;
        const double *vals = static_cast<const double *>(dvals.p);
        const int32_t *rowptr = static_cast<const int32_t *>(drowptr.p), *col = static_cast<const int32_t *>(dcol.p);
        double *Minv = static_cast<double *>(dminv.p), *x = static_cast<double *>(dx.p), *r = static_cast<double *>(dr.p);
        double *z = static_cast<double *>(dz.p), *q = static_cast<double *>(dq.p);
        double *pq = static_cast<double *>(dpart.p), *prz = pq + ctx->sm_count * spg::PCG_CTAS_PER_SM;
        double *prr = prz + ctx->sm_count * spg::PCG_CTAS_PER_SM;
        double *pa = static_cast<double *>(dp0.p), *pb = static_cast<double *>(dp1.p);
        spg::PcgState *state = static_cast<spg::PcgState *>(dstate.p);
        SPG_CUDA(cudaMemsetAsync(state, 0, sizeof(spg::PcgState), st));
        SPG_CUDA(cudaMemsetAsync(pa, 0, (size_t) n * 8, st)); // p_0 = z_0 + 0 * pa
        spg::bsr_block_jacobi_kernel<D><<<grid_rows, 256, 0, st>>>(vals, static_cast<const int32_t *>(ddiag.p), nb, lambda, Minv, state);
        spg::pcg_update_kernel<D><<<grid_rows, 256, 0, st>>>(nb, true, Minv, g, pa, q, x, r, z, state, prz, prr);
        spg::pcg_beta_kernel<<<1, 1024, 0, st>>>(prz, prr, grid_rows, true, spg::PCG_TOL, spg::PCG_MAX_ITERS, state);
        ctx->launches += 3;
        spg::PcgState h{};
        for(;;) {
            for(int k = 0; k < spg::PCG_POLL; k++) {
                spg::pcg_spmv_dot_kernel<D><<<grid_spmv, 256, 0, st>>>(nb, rowptr, col, vals, lambda, z, pa, pb, q, state, pq);
                spg::pcg_alpha_kernel<<<1, 1024, 0, st>>>(pq, grid_spmv, state);
                spg::pcg_update_kernel<D><<<grid_rows, 256, 0, st>>>(nb, false, Minv, g, pb, q, x, r, z, state, prz, prr);
                spg::pcg_beta_kernel<<<1, 1024, 0, st>>>(prz, prr, grid_rows, false, spg::PCG_TOL, spg::PCG_MAX_ITERS, state);
                std::swap(pa, pb);
            }
            ctx->launches += 4 * spg::PCG_POLL;
            SPG_CUDA(cudaMemcpyAsync(&h, state, sizeof(h), cudaMemcpyDeviceToHost, st));
            SPG_CUDA(cudaStreamSynchronize(st));
            if(h.done) break;
        }
        SPG_CUDA(cudaGetLastError());
        SPG_CUDA(cudaMemcpyAsync(hx.data(), x, (size_t) n * 8, cudaMemcpyDeviceToHost, st));
        SPG_CUDA(cudaStreamSynchronize(st));
        cg_iterations += h.iters;
        cg_max_rel_residual = std::max(cg_max_rel_residual, h.rel);
        *ok = !h.bad;
        if(!*ok) std::fill(hx.begin(), hx.end(), 0.0); // the trial is rejected; keep computeScale finite
        return SPG_OK;
    }
};

struct LmResult {
    int iterations = 0, trials = 0;
    bool terminated = false;
    double chi2_initial = 0, chi2 = 0, lambda = 0;
};

// GraphWrapperG2O::optimize (:250-269) with g2o's OptimizationAlgorithmLevenberg (default parameters) on the poses of
// dg, which are uploaded in arr and updated in both. g: n doubles, sc: 2 doubles of device scratch.
spg_status levenberg_marquardt(spg_ctx *ctx, DeviceGraph &dg, DevArrays &arr, const std::vector<int32_t> &pos, int n,
                               int max_iterations, LinearSystem &sys, double *g, double *sc, LmResult &res) {
    cudaStream_t st = ctx->stream;
    auto push_poses = [&]() -> cudaError_t {
        return cudaMemcpyAsync(arr.poses.p, dg.poses.data(), dg.poses.size() * 8, cudaMemcpyHostToDevice, st);
    };
    auto chi2_only = [&](double *out) -> spg_status {
        spg_status s = assemble(ctx, dg, arr, n, nullptr, n, nullptr, sc);
        if(s != SPG_OK) return s;
        SPG_CUDA(cudaMemcpyAsync(out, sc, 8, cudaMemcpyDeviceToHost, st));
        SPG_CUDA(cudaStreamSynchronize(st));
        return SPG_OK;
    };
#define SPG_TRY(call)           \
    do {                        \
        spg_status s_ = (call); \
        if(s_ != SPG_OK) return s_; \
    } while(0)
    const size_t nn = (size_t) std::max(n, 1);
    std::vector<double> hx(nn), hg(nn), saved;
    double lambda = 0, ni = 2, chi = 0;
    int iters = 0, trials_total = 0;
    bool terminated = false;
    SPG_TRY(chi2_only(&chi));
    const double chi_initial = chi;
    for(int it = 0; it < max_iterations && n > 0 && !terminated; it++) {
        // buildSystem at the current estimates
        SPG_TRY(sys.build(g, sc));
        if(it == 0) { // computeLambdaInit: tau * max diagonal entry, tau = 1e-5
            SPG_TRY(sys.max_diag(sc + 1));
            double md = 0;
            SPG_CUDA(cudaMemcpyAsync(&md, sc + 1, 8, cudaMemcpyDeviceToHost, st));
            SPG_CUDA(cudaStreamSynchronize(st));
            lambda = 1e-5 * md;
            ni = 2;
        }
        SPG_CUDA(cudaMemcpyAsync(hg.data(), g, (size_t) n * 8, cudaMemcpyDeviceToHost, st));
        double rho = 0;
        int qmax = 0;
        saved = dg.poses;
        do {
            // (H + lambda I) x = -g   [g2o: b = -J^T Omega e]
            bool ok2 = false;
            SPG_TRY(sys.solve(lambda, g, hg, hx, &ok2));
            // update (push / oplus)
            if(ok2)
                for(int v = 0; v < dg.nV; v++)
                    if(pos[v] >= 0) oplus_flat(dg.dim, &dg.poses[(size_t) v * dg.P], &hx[pos[v]]);
            SPG_CUDA(push_poses());
            double tempChi = 0;
            SPG_TRY(chi2_only(&tempChi));
            if(!ok2) tempChi = std::numeric_limits<double>::max();
            rho = chi - tempChi;
            double scale = 0; // computeScale: sum x_j (lambda x_j + b_j), b = -g
            for(int q = 0; q < n; q++) scale += hx[q] * (lambda * hx[q] - hg[q]);
            scale += 1e-3;
            rho /= scale;
            if(rho > 0 && std::isfinite(tempChi)) { // last step was good
                double alpha = 1.0 - std::pow(2 * rho - 1, 3);
                alpha = std::min(alpha, 2.0 / 3.0);
                lambda *= std::max(1.0 / 3.0, alpha);
                ni = 2;
                chi = tempChi;
            } else {
                lambda *= ni;
                ni *= 2;
                dg.poses = saved; // pop
                SPG_CUDA(push_poses());
                if(!std::isfinite(lambda)) break;
            }
            qmax++;
            trials_total++;
        } while(rho < 0 && qmax < 10);
        iters++;
        if(qmax == 10 || rho == 0 || !std::isfinite(lambda)) terminated = true;
    }
#undef SPG_TRY
    SPG_CUDA(cudaStreamSynchronize(st));
    res.iterations = iters;
    res.trials = trials_total;
    res.terminated = terminated;
    res.chi2_initial = chi_initial;
    res.chi2 = chi;
    res.lambda = lambda;
    return SPG_OK;
}

// Largest system the dense path takes: two n x n buffers of 8-byte words, 120 GB for H, as before the sparse path. The
// environment variable SPG_OPT_DENSE_MAX_DIMS lowers it (tests: the sparse path on graphs the dense path also solves);
// read on every call so it can be set after the library is loaded.
bool dense_fits(int n) {
    if((double) n * n * 8 > 120e9) return false;
    const char *e = getenv("SPG_OPT_DENSE_MAX_DIMS");
    return !(e && *e && n > atoll(e));
}

} // namespace

extern "C" {

spg_status spg_graph_kld(spg_ctx *ctx, const spg_graph *full, const spg_graph *sparse, int32_t fixed_id, double *kld, spg_kld_terms *terms) {
    if(!ctx || !full || !sparse || !kld || full->g->dim != sparse->g->dim) {
        spg_set_err("spg_graph_kld: bad arguments");
        return SPG_ERR_INVALID;
    }
    SPG_CUDA(cudaSetDevice(ctx->device));
    SPG_CUDA(configure_dense());
    DeviceGraph F, S;
    flatten(*full->g, F);
    flatten(*sparse->g, S);
    const int dim = F.dim;
    // computeIndices (:472-499): the variables of the sparsified graph are kept, the rest of the full graph is marginalised
    std::vector<char> fixedF(F.nV, 0), keepF(F.nV, 0), fixedS(S.nV, 0);
    {
        size_t j = 0;
        for(int i = 0; i < F.nV; i++) {
            if(F.ids[i] == fixed_id) fixedF[i] = 1;
            while(j < S.ids.size() && S.ids[j] < F.ids[i]) j++;
            if(j < S.ids.size() && S.ids[j] == F.ids[i]) keepF[i] = 1;
        }
        for(int i = 0; i < S.nV; i++) {
            if(S.ids[i] == fixed_id) fixedS[i] = 1;
            if(!std::binary_search(F.ids.begin(), F.ids.end(), S.ids[i])) {
                spg_set_err("spg_graph_kld: vertex " + std::to_string(S.ids[i]) + " of the sparsified graph is not in the full graph");
                return SPG_ERR_INVALID;
            }
        }
    }
    std::vector<int32_t> posF, posS;
    int nm = 0;
    const int nf = layout(F, fixedF, &keepF, posF, &nm);
    const int nk = layout(S, fixedS, nullptr, posS, nullptr);
    if(nf - nm != nk || nk == 0) {
        spg_set_err("spg_graph_kld: kept dimensions of the two graphs differ");
        return SPG_ERR_INVALID;
    }
    const double bytes = ((double) nf * nf + 2.0 * nk * nk) * 8;
    if(bytes > 120e9) {
        spg_set_err("spg_graph_kld: dense evaluation needs " + std::to_string((long long) (bytes / 1e9)) + " GB");
        return SPG_ERR_UNSUPPORTED;
    }
    // estimateDifference (:550-575) on the kept vertices, in the sparsified graph's order
    std::vector<double> diff((size_t) nk, 0.0);
    for(int i = 0, k = 0; i < S.nV; i++) {
        if(fixedS[i]) continue;
        const int fi = (int) (std::lower_bound(F.ids.begin(), F.ids.end(), S.ids[i]) - F.ids.begin());
        const double *a = &F.poses[(size_t) fi * F.P], *b = &S.poses[(size_t) i * S.P];
        if(dim == 3) {
            diff[k] = a[0] - b[0];
            diff[k + 1] = a[1] - b[1];
            double th = a[2] - b[2];
            while(th > M_PI) th -= 2 * M_PI;
            while(th < -M_PI) th += 2 * M_PI;
            diff[k + 2] = th;
        } else {
            double inv[7], rel[7];
            spg::poseInverse(6, a, inv);
            spg::poseCompose(6, inv, b, rel);
            const double sgn = rel[6] < 0 ? -1.0 : 1.0; // CondensedQuaternion: w >= 0
            for(int q = 0; q < 3; q++) diff[k + q] = rel[q];
            for(int q = 0; q < 3; q++) diff[k + 3 + q] = sgn * rel[3 + q];
        }
        k += dim;
    }

    cudaStream_t st = ctx->stream;
    cudaEvent_t e0, e1;
    SPG_CUDA(cudaEventCreate(&e0));
    SPG_CUDA(cudaEventCreate(&e1));
    DevBuf dHf, dHs, dLx, dsc, dd;
    DevArrays aF, aS;
    auto cleanup = [&] {
        for(DevBuf *b : {&dHf, &dHs, &dLx, &dsc, &dd}) b->release();
        release(aF);
        release(aS);
        cudaEventDestroy(e0);
        cudaEventDestroy(e1);
    };
#define SPG_TRY(call)                    \
    do {                                 \
        spg_status s_ = (call);          \
        if(s_ != SPG_OK) {               \
            cleanup();                   \
            return s_;                   \
        }                                \
    } while(0)
#define SPG_CUDA_C(call)                                                            \
    do {                                                                            \
        cudaError_t e_ = (call);                                                    \
        if(e_ != cudaSuccess) {                                                     \
            spg_set_err(std::string(#call) + ": " + cudaGetErrorString(e_));        \
            cleanup();                                                              \
            return SPG_ERR_CUDA;                                                    \
        }                                                                           \
    } while(0)
    SPG_CUDA_C(dHf.reserve((size_t) nf * nf * 8));
    SPG_CUDA_C(dHs.reserve((size_t) nk * nk * 8));
    SPG_CUDA_C(dLx.reserve((size_t) nk * nk * 8));
    SPG_CUDA_C(dsc.reserve(64)); // [0] logdet_m [1] logdet_y [2] logdet_x [3] innerprod [4] maha, flags at +48
    SPG_CUDA_C(dd.reserve((size_t) nk * 8));
    double *Hf = static_cast<double *>(dHf.p), *Hs = static_cast<double *>(dHs.p), *Lx = static_cast<double *>(dLx.p);
    double *sc = static_cast<double *>(dsc.p);
    int *flags = reinterpret_cast<int *>(sc + 6);
    SPG_CUDA_C(cudaMemsetAsync(sc, 0, 64, st));
    SPG_CUDA_C(cudaMemcpyAsync(dd.p, diff.data(), (size_t) nk * 8, cudaMemcpyHostToDevice, st));
    SPG_TRY(upload(ctx, F, posF, aF));
    SPG_TRY(upload(ctx, S, posS, aS));
    SPG_CUDA_C(cudaEventRecord(e0, st));
    SPG_TRY(assemble(ctx, F, aF, nf, Hf, nf, nullptr, nullptr));
    SPG_TRY(assemble(ctx, S, aS, nk, Hs, nk, nullptr, nullptr));
    // Lambda_y: Schur complement of the full information onto the kept variables (:539-542)
    cholesky_partial(ctx, Hf, nf, nf, nm, sc + 0, flags + 0);
    double *Ly = Hf + nm + (int64_t) nm * nf; // nk x nk, leading dimension nf, lower triangle
    // Mahalanobis term with Lambda_x before it is factorised (utils.cpp:88)
    spg::quad_form_lower_kernel<<<ctx->sm_count * 4, 256, 0, st>>>(Hs, nk, nk, static_cast<const double *>(dd.p), sc + 4);
    SPG_CUDA_C(cudaMemcpyAsync(Lx, Hs, (size_t) nk * nk * 8, cudaMemcpyDeviceToDevice, st));
    cholesky_partial(ctx, Lx, nk, nk, nk, sc + 2, flags + 1); // Lambda_x = Lx Lx^T, logdet_x
    cholesky_partial(ctx, Ly, nf, nk, nk, sc + 1, flags + 2); // Lambda_y = Ly Ly^T, logdet_y
    // tr(Lambda_y^-1 Lambda_x) = || Ly^-1 Lx ||_F^2
    spg::zero_upper_kernel<<<(unsigned) (((int64_t) nk * nk + 255) / 256), 256, 0, st>>>(Lx, nk, nk);
    forward_solve(ctx, Ly, nf, nk, Lx, nk, nk);
    spg::frob2_lower_kernel<<<ctx->sm_count * 4, 256, 0, st>>>(Lx, nk, nk, sc + 3);
    ctx->launches += 3;
    SPG_CUDA_C(cudaEventRecord(e1, st));
    double h[8];
    SPG_CUDA_C(cudaMemcpyAsync(h, sc, 64, cudaMemcpyDeviceToHost, st));
    SPG_CUDA_C(cudaStreamSynchronize(st));
    SPG_CUDA_C(cudaGetLastError());
    float ms = 0;
    cudaEventElapsedTime(&ms, e0, e1);
    int hf[4];
    std::memcpy(hf, h + 6, sizeof(int) * 4);
    cleanup();
#undef SPG_TRY
#undef SPG_CUDA_C
    if(hf[0] || hf[1] || hf[2]) {
        spg_set_err(std::string("spg_graph_kld: information matrix not positive definite (") +
                    (hf[0] ? "marginalised block of the full graph" : hf[1] ? "sparsified graph" : "marginal of the full graph") + ")");
        return SPG_ERR_INVALID;
    }
    // utils.cpp:92: kld = 1/2 (innerprod + mahalanobis - logdetx - logdety - n) with logdety = -logdet(Lambda_y)
    const double logdet_y = h[1], logdet_x = h[2], inner = h[3], maha = h[4];
    *kld = 0.5 * (inner + maha - logdet_x + logdet_y - nk);
    if(terms) {
        terms->innerprod = inner;
        terms->mahalanobis = maha;
        terms->logdet_x = logdet_x;
        terms->logdet_y = logdet_y;
        terms->n_keep = nk;
        terms->n_marginalized = nm;
        terms->device_ms = ms;
        terms->flops = ((double) nf * nf * nf - (double) nk * nk * nk) / 3.0 + 2.0 * (double) nk * nk * nk / 3.0 + (double) nk * nk * nk / 3.0;
    }
    return SPG_OK;
}

// GraphWrapperG2O::optimize (:250-269) with g2o's OptimizationAlgorithmLevenberg (default parameters). fixed_ids: the
// vertices held fixed (the reference fixes vertex 0; chi2(other) fixes other's vertices). Dense Cholesky wherever the
// dense system fits; block-sparse PCG beyond that.
spg_status spg_graph_optimize(spg_ctx *ctx, spg_graph *gr, const int32_t *fixed_ids, int32_t n_fixed, int32_t max_iterations,
                              spg_optimize_stats *stats) {
    if(!ctx || !gr || n_fixed < 0 || (n_fixed > 0 && !fixed_ids) || max_iterations < 0) {
        spg_set_err("spg_graph_optimize: bad arguments");
        return SPG_ERR_INVALID;
    }
    SPG_CUDA(cudaSetDevice(ctx->device));
    SPG_CUDA(configure_dense());
    Graph &G = *gr->g;
    DeviceGraph dg;
    flatten(G, dg);
    std::vector<char> fixed(dg.nV, 0);
    for(int i = 0; i < n_fixed; i++) {
        auto it = std::lower_bound(dg.ids.begin(), dg.ids.end(), fixed_ids[i]);
        if(it != dg.ids.end() && *it == fixed_ids[i]) fixed[it - dg.ids.begin()] = 1;
    }
    std::vector<int32_t> pos;
    const int n = layout(dg, fixed, nullptr, pos, nullptr);
    if(stats) *stats = spg_optimize_stats{};
    DevBuf dg_, dsc;
    DevArrays arr;
    Bsr bsr;
    std::unique_ptr<DenseSystem> dense;
    std::unique_ptr<SparseSystem> sparse;
    auto cleanup = [&] {
        dense.reset();
        sparse.reset();
        for(DevBuf *b : {&dg_, &dsc}) b->release();
        release(arr);
    };
#define SPG_CUDA_C(call)                                                            \
    do {                                                                            \
        cudaError_t e_ = (call);                                                    \
        if(e_ != cudaSuccess) {                                                     \
            spg_set_err(std::string(#call) + ": " + cudaGetErrorString(e_));        \
            cleanup();                                                              \
            return SPG_ERR_CUDA;                                                    \
        }                                                                           \
    } while(0)
#define SPG_TRY(call)                    \
    do {                                 \
        spg_status s_ = (call);          \
        if(s_ != SPG_OK) {               \
            cleanup();                   \
            return s_;                   \
        }                                \
    } while(0)
    if(dense_fits(n)) {
        dense.reset(new DenseSystem(ctx, dg, arr, n));
        const cudaError_t e = dense->reserve();
        if(e == cudaErrorMemoryAllocation) { // not enough free HBM for the two dense buffers: go sparse
            cudaGetLastError();
            dense.reset();
        } else {
            SPG_CUDA_C(e);
        }
    }
    const size_t nn = (size_t) std::max(n, 1);
    SPG_CUDA_C(dg_.reserve(nn * 8));
    SPG_CUDA_C(dsc.reserve(64));
    if(!dense) {
        SPG_TRY(build_bsr(dg, pos, n, bsr));
        sparse.reset(new SparseSystem(ctx, dg, arr, bsr, n));
        SPG_TRY(sparse->reserve());
    }
    SPG_TRY(upload(ctx, dg, pos, arr, dense ? nullptr : &bsr));
    LinearSystem &sys = dense ? static_cast<LinearSystem &>(*dense) : static_cast<LinearSystem &>(*sparse);
    LmResult res;
    SPG_TRY(levenberg_marquardt(ctx, dg, arr, pos, n, max_iterations, sys, static_cast<double *>(dg_.p),
                                static_cast<double *>(dsc.p), res));
    const bool used_dense = dense != nullptr;
    const int64_t cg_iterations = sys.cg_iterations;
    const double cg_max_rel = sys.cg_max_rel_residual;
    cleanup();
#undef SPG_CUDA_C
#undef SPG_TRY
    // write the estimates back
    for(int v = 0; v < dg.nV; v++) {
        spg::GraphVertex *gv = G.vertex(dg.ids[v]);
        std::memcpy(gv->pose, &dg.poses[(size_t) v * dg.P], sizeof(double) * dg.P);
    }
    G.version++;
    if(stats) {
        stats->iterations = res.iterations;
        stats->trials = res.trials;
        stats->dimensions = n;
        stats->chi2_initial = res.chi2_initial;
        stats->chi2_final = res.chi2;
        stats->lambda_final = res.lambda;
        stats->terminated = res.terminated ? 1 : 0;
        stats->solver = used_dense ? SPG_SOLVER_DENSE_CHOLESKY : SPG_SOLVER_SPARSE_PCG;
        stats->cg_iterations = (int32_t) std::min<int64_t>(cg_iterations, std::numeric_limits<int32_t>::max());
        stats->cg_max_rel_residual = cg_max_rel;
    }
    return SPG_OK;
}

spg_status spg_graph_chi2(spg_ctx *ctx, const spg_graph *gr, double *chi2) {
    if(!ctx || !gr || !chi2) return SPG_ERR_INVALID;
    SPG_CUDA(cudaSetDevice(ctx->device));
    DeviceGraph dg;
    flatten(*gr->g, dg);
    std::vector<int32_t> pos((size_t) dg.nV, -1);
    DevArrays arr;
    DevBuf dsc;
    spg_status s = upload(ctx, dg, pos, arr);
    if(s == SPG_OK && dsc.reserve(16) != cudaSuccess) s = SPG_ERR_CUDA;
    if(s == SPG_OK) s = assemble(ctx, dg, arr, 0, nullptr, 1, nullptr, static_cast<double *>(dsc.p));
    if(s == SPG_OK) {
        if(cudaMemcpyAsync(chi2, dsc.p, 8, cudaMemcpyDeviceToHost, ctx->stream) != cudaSuccess ||
           cudaStreamSynchronize(ctx->stream) != cudaSuccess)
            s = SPG_ERR_CUDA;
    }
    release(arr);
    dsc.release();
    return s;
}

} // extern "C"
