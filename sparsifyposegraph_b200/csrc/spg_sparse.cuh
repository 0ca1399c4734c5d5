// spg_sparse.cuh — block-sparse (BSR) linear algebra of spg_graph_optimize for graphs whose dense system does not fit:
// (H + lambda I) x = -g by preconditioned conjugate gradients with a block-Jacobi preconditioner (g2o's
// LinearSolverPCG). H is stored in both triangles, one D x D column-major block per slot, so the product runs one block
// row per warp without atomics. Every reduction is fixed-order (per-CTA partials, then one single-CTA pass), so a solve
// adds no run-to-run variation of its own.
#pragma once
#include <cstdint>

namespace spg {

// Stopping rule: ||r|| <= PCG_TOL ||b||. The LM step is a Newton step: a relative residual of 1e-6 leaves the step
// error about six orders below the step, far below what the rho test can see, and LM re-linearises anyway, so a
// tighter solve buys nothing.
constexpr double PCG_TOL = 1e-6;
// Iteration cap. A 2-D grid of width w anchored at one vertex needs O(w) block-Jacobi CG iterations per digit; 5000
// reaches 1e-6 on grids of ~1000 poses a side. A trial that hits the cap still proposes its step, and LM's rho test
// judges it like any other.
constexpr int PCG_MAX_ITERS = 5000;
// The host reads the done flag every PCG_POLL iterations; iterations after the rule holds are no-ops on the device.
constexpr int PCG_POLL = 32;
constexpr int PCG_CTAS_PER_SM = 16; // grid bound of the row kernels, and so the length of the partial-sum arrays

struct PcgState {
    double rz, bb, alpha, beta, rel; // r.z, ||b||^2, step lengths, ||r|| / ||b|| at the last reduction
    int32_t done, iters, bad, pad;   // bad: a diagonal block or p.Ap not positive (H + lambda I not positive definite)
};

// sum of a[0 .. n) in a fixed order, result in thread 0 (one CTA of 1024 threads)
__device__ __forceinline__ double cta_sum_fixed(const double *a, int n) {
    __shared__ double sh[32];
    double s = 0;
    for(int i = threadIdx.x; i < n; i += blockDim.x) s += a[i];
    for(int o = 16; o > 0; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o);
    __syncthreads();
    if((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = s;
    __syncthreads();
    if(threadIdx.x == 0)
        for(int w = 1; w < (int) (blockDim.x >> 5); w++) s += sh[w];
    return s;
}

// per-CTA sum of one value per thread, fixed order, written by thread 0 to out[blockIdx.x]
__device__ __forceinline__ void cta_partial(double v, double *out) {
    __shared__ double sh[32];
    for(int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    if((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
    __syncthreads();
    if(threadIdx.x == 0) {
        for(int w = 1; w < (int) (blockDim.x >> 5); w++) v += sh[w];
        out[blockIdx.x] = v;
    }
}

// largest diagonal entry of H (computeLambdaInit); single CTA
template <int D>
__global__ void bsr_max_diag_kernel(const double *vals, const int32_t *diag, int nb, double *out) {
    double m = 0;
    for(int i = threadIdx.x; i < nb * D; i += blockDim.x) m = fmax(m, vals[(int64_t) diag[i / D] * D * D + (i % D) * (D + 1)]);
    for(int o = 16; o > 0; o >>= 1) m = fmax(m, __shfl_down_sync(0xffffffffu, m, o));
    __shared__ double part[32];
    if((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = m;
    __syncthreads();
    if(threadIdx.x == 0) {
        for(int w = 1; w < (int) (blockDim.x >> 5); w++) m = fmax(m, part[w]);
        *out = m;
    }
}

// Minv_i = (H_ii + lambda I)^-1 by a Cholesky of the D x D block; one thread per block row
template <int D>
__global__ void bsr_block_jacobi_kernel(const double *vals, const int32_t *diag, int nb, double lambda, double *Minv, PcgState *st) {
    for(int i = blockIdx.x * blockDim.x + threadIdx.x; i < nb; i += gridDim.x * blockDim.x) {
        const double *B = vals + (int64_t) diag[i] * D * D;
        double L[D * D];
        for(int k = 0; k < D * D; k++) L[k] = B[k];
        for(int k = 0; k < D; k++) L[k * (D + 1)] += lambda;
        bool ok = true;
        for(int j = 0; j < D; j++) { // lower factor in place, column-major
            double d = L[j + j * D];
            for(int k = 0; k < j; k++) d -= L[j + k * D] * L[j + k * D];
            ok = ok && d > 0 && isfinite(d);
            d = sqrt(fmax(d, 1e-300));
            L[j + j * D] = d;
            for(int r = j + 1; r < D; r++) {
                double s = L[r + j * D];
                for(int k = 0; k < j; k++) s -= L[r + k * D] * L[j + k * D];
                L[r + j * D] = s / d;
            }
        }
        if(!ok) st->bad = 1;
        double *M = Minv + (int64_t) i * D * D;
        for(int c = 0; c < D; c++) { // column c of (L L^T)^-1: L y = e_c, L^T x = y
            double y[D];
            for(int r = 0; r < D; r++) {
                double s = r == c ? 1.0 : 0.0;
                for(int k = 0; k < r; k++) s -= L[r + k * D] * y[k];
                y[r] = s / L[r + r * D];
            }
            for(int r = D - 1; r >= 0; r--) {
                double s = y[r];
                for(int k = r + 1; k < D; k++) s -= L[k + r * D] * y[k];
                y[r] = s / L[r + r * D];
            }
            for(int r = 0; r < D; r++) M[r + c * D] = y[r];
        }
    }
}

// p = z + beta p_old (written for the warp's own rows to p_new, formed on the fly for its columns), q = (H + lambda I) p,
// partial sums of p.q; one warp per block row
template <int D>
__global__ void __launch_bounds__(256) pcg_spmv_dot_kernel(int nb, const int32_t *rowptr, const int32_t *col, const double *vals,
                                                           double lambda, const double *z, const double *p_old, double *p_new,
                                                           double *q, const PcgState *st, double *partial) {
    if(st->done) return;
    constexpr int G = 32 / D; // slots of a row in flight per warp, D lanes (one per block row entry) each
    __shared__ double sh[8][32];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, g = lane / D, rr = lane % D;
    const double beta = st->beta;
    double dot = 0;
    for(int i = blockIdx.x * 8 + w; i < nb; i += gridDim.x * 8) {
        double acc = 0;
        if(g < G)
            for(int s = rowptr[i] + g; s < rowptr[i + 1]; s += G) {
                const double *B = vals + (int64_t) s * D * D;
                const int64_t j = (int64_t) col[s] * D;
#pragma unroll
                for(int c = 0; c < D; c++) acc += B[rr + c * D] * (z[j + c] + beta * p_old[j + c]);
            }
        sh[w][lane] = acc;
        __syncwarp();
        if(lane < D) {
            double y = 0;
            for(int k = 0; k < G; k++) y += sh[w][k * D + lane];
            const int64_t e = (int64_t) i * D + lane;
            const double pi = z[e] + beta * p_old[e];
            y += lambda * pi;
            p_new[e] = pi;
            q[e] = y;
            dot += pi * y;
        }
        __syncwarp();
    }
    cta_partial(dot, partial);
}

// init: x = 0, r = -g; otherwise x += alpha p, r -= alpha q. Then z = Minv r and partial sums of r.z and r.r;
// one thread per block row
template <int D>
__global__ void __launch_bounds__(256) pcg_update_kernel(int nb, bool init, const double *Minv, const double *g, const double *p,
                                                         const double *q, double *x, double *r, double *z, const PcgState *st,
                                                         double *partial_rz, double *partial_rr) {
    if(st->done) return;
    const double alpha = st->alpha;
    double rz = 0, rr = 0;
    for(int i = blockIdx.x * blockDim.x + threadIdx.x; i < nb; i += gridDim.x * blockDim.x) {
        const int64_t e = (int64_t) i * D;
        double ri[D];
        for(int k = 0; k < D; k++) {
            if(init) {
                x[e + k] = 0;
                ri[k] = -g[e + k];
            } else {
                x[e + k] += alpha * p[e + k];
                ri[k] = r[e + k] - alpha * q[e + k];
            }
            r[e + k] = ri[k];
            rr += ri[k] * ri[k];
        }
        const double *M = Minv + (int64_t) i * D * D;
        for(int k = 0; k < D; k++) {
            double s = 0;
            for(int c = 0; c < D; c++) s += M[k + c * D] * ri[c];
            z[e + k] = s;
            rz += ri[k] * s;
        }
    }
    cta_partial(rz, partial_rz);
    __syncthreads();
    cta_partial(rr, partial_rr);
}

// alpha = r.z / p.Ap; single CTA of 1024 threads
__global__ void __launch_bounds__(1024) pcg_alpha_kernel(const double *partial, int n, PcgState *st) {
    if(st->done) return;
    const double pq = cta_sum_fixed(partial, n);
    if(threadIdx.x == 0) {
        if(!(pq > 0) || !isfinite(pq)) {
            st->bad = 1;
            st->done = 1;
        } else {
            st->alpha = st->rz / pq;
        }
    }
}

// beta = r.z (new) / r.z (old) and the stopping rule; with `init` the start of a solve (||b||^2, beta = 0).
// Single CTA of 1024 threads.
__global__ void __launch_bounds__(1024) pcg_beta_kernel(const double *partial_rz, const double *partial_rr, int n, bool init,
                                                        double tol, int max_iters, PcgState *st) {
    if(st->done) return;
    const double rz = cta_sum_fixed(partial_rz, n);
    __syncthreads();
    const double rr = cta_sum_fixed(partial_rr, n);
    if(threadIdx.x != 0) return;
    if(init) {
        st->bb = rr;
        st->beta = 0;
        st->iters = 0;
    } else {
        st->beta = rz / st->rz;
        st->iters++;
    }
    st->rz = rz;
    st->rel = st->bb > 0 ? sqrt(rr / st->bb) : 0.0;
    if(st->rel <= tol || st->iters >= max_iters || st->bad) st->done = 1;
}

} // namespace spg
