// spg_fast.cuh — the NFR-tree kernel (sm_100a): the path BASELINE.json's metric is quoted on and the one the
// shipped datasets take (Chow-Liu tree + closed-form information fit), for blankets of relative-pose edges with
// one removed vertex. Same stages as blanket_kernel (spg_kernels.cuh) — assembly, Schur complement, Chow-Liu,
// gauge shortcut, closed form (reference src/vertex_remover.cpp:394-450, src/pseudo_chow_liu.cpp,
// src/logdet_function.cpp:236-279) — built around ONE data structure: the symmetric k x k matrix of the kept
// variables lives in REGISTERS from the assembly to the last sweep, as D x D blocks of its lower block triangle,
// one (row vertex, column vertex) block per thread.
//   * H_kk is accumulated straight into the blocks (no N x N matrix anywhere), the rank-d Schur update is applied
//     in registers, and both SPD inverses (C = (Lambda_t + I)^-1 and the anchored G = Lambda_rr^-1) are symmetric
//     Gauss-Jordan sweeps over the lower block triangle: half the FMAs and half the threads of a full-matrix
//     sweep. Per pivot only the pivot column crosses shared memory (double buffered, one barrier, look-ahead).
//   * No k x k matrix is ever stored in shared memory: the Chow-Liu weights are computed by the thread that holds
//     the block C_ji (diagonal blocks are published, 36 doubles per vertex), the Sigma blocks of the closed form
//     are scattered from the registers that hold G. A 16-vertex SE3 blanket needs 120 threads and ~53 KB instead
//     of 256 threads and 229.7 KB: FOUR blankets per SM (four independent pivot chains) instead of one; a
//     blanket of <= 8 vertices is ONE warp with __syncwarp() as its only barrier, 10-16 blankets per SM.
//   * The kernel carries nothing but this path (no GLC, no Newton loop, no Jacobi eigen-solver). Whatever it does
//     not take — GLC / MULTI input edges, several removed vertices, a refused gauge guard, any non-positive
//     pivot — is appended to a device-side retry list and re-run by blanket_kernel, which reports the status.
#pragma once
#include "spg_kernels.cuh"

namespace spg {

template <bool ONEWARP>
__device__ __forceinline__ void fsync() {
    if constexpr(ONEWARP) __syncwarp();
    else __syncthreads();
}
template <bool ONEWARP>
__device__ __forceinline__ int fsync_or(int pred) {
    if constexpr(ONEWARP) return __any_sync(0xffffffffu, pred);
    else return __syncthreads_or(pred);
}
// sum over the CTA in a fixed order; every thread gets the result. red: >= 32 doubles.
template <bool ONEWARP>
__device__ __forceinline__ double fsum(double v, double *red) {
#pragma unroll
    for(int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if constexpr(ONEWARP) return v;
    else {
        const int w = threadIdx.x >> 5, l = threadIdx.x & 31, nw = (blockDim.x + 31) >> 5;
        __syncthreads();
        if(l == 0) red[w] = v;
        __syncthreads();
        double s = 0;
        for(int i = 0; i < nw; i++) s += red[i];
        return s;
    }
}

// Thread group that owns one blanket. G = 8 / 16 / 32: a sub-warp group of G lanes (32 / G blankets per warp side
// by side, each group with its own control flow, shared-memory slot and masked warp barriers; a CTA is one or
// several such warps, see the phase barriers of fast_kernel); G = 0: the whole CTA (blockDim.x threads,
// __syncthreads).
template <int G>
struct Grp {
    static __device__ __forceinline__ unsigned mask() {
        if constexpr(G == 32 || G == 0) return 0xffffffffu;
        else return ((1u << G) - 1u) << (G * ((threadIdx.x & 31) / G));
    }
    static __device__ __forceinline__ int tid() { return G ? (int) (threadIdx.x % (G ? G : 1)) : (int) threadIdx.x; }
    static __device__ __forceinline__ int nt() { return G ? G : (int) blockDim.x; }
    static __device__ __forceinline__ int slot() { return G ? (int) (threadIdx.x / (G ? G : 1)) : 0; }
    static __device__ __forceinline__ int slots() { return G ? (int) blockDim.x / (G ? G : 1) : 1; }
    static __device__ __forceinline__ void sync() {
        if constexpr(G == 0) __syncthreads();
        else __syncwarp(mask());
    }
    static __device__ __forceinline__ int any(int pred) {
        if constexpr(G == 0) return __syncthreads_or(pred);
        else return __any_sync(mask(), pred);
    }
    // sum in a fixed order; every thread of the group gets the result. red: >= 32 doubles (G = 0 only)
    static __device__ __forceinline__ double sum(double v, double *red) {
        if constexpr(G == 0) {
#pragma unroll
            for(int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
            const int w = threadIdx.x >> 5, l = threadIdx.x & 31, nw = (blockDim.x + 31) >> 5;
            __syncthreads();
            if(l == 0) red[w] = v;
            __syncthreads();
            double s = 0;
            for(int i = 0; i < nw; i++) s += red[i];
            return s;
        } else {
            const unsigned m = mask();
#pragma unroll
            for(int o = G / 2; o > 0; o >>= 1) v += __shfl_xor_sync(m, v, o);
            return v;
        }
    }
};

// ---- block sweep ---------------------------------------------------------------------------------------------
// The symmetric sweep operator (B_jj = -1/d, B_ij = A_ij / d, B_il = A_il - A_ij A_jl / d; all pivots swept: -A^-1)
// applied one VERTEX (D pivots) at a time on the D x D register blocks of the lower block triangle. Per vertex J:
//   (a) the thread of the diagonal block inverts it in registers (D scalar sweep steps, the pivots are the scalar
//       sweep's pivots: pivot > 0 is LLT's positive-definiteness test) and publishes B = A_JJ^-1;
//   (c) the threads of block column J (below the diagonal) and block row J (left of it) publish their panel block
//       P_I = A_IJ and W_I = P_I B, and keep W_I (the swept panel) as their block;
//   (e) every other block (I, L) -= W_I P_L^T: 6 x 36 independent DFMAs per thread, operands by 16-byte loads from
//       shared memory; the thread of the next diagonal block goes on with (a) for vertex J + 1.
// Two barriers per vertex instead of one per pivot, and two thirds of the instructions of a pivot-by-pivot sweep.
template <int D> struct FastPad { static constexpr int PST = (D * D + 3) & ~1; }; // panel block stride: 38 (SE3), 10 (SE2)

template <int D>
__device__ __forceinline__ void invert_tile(double (&a)[D][D], double *Bout, double *piv, bool &bad) {
#pragma unroll
    for(int s = 0; s < D; s++) {
        const double d = a[s][s];
        bad |= !(d > 0);
        piv[s] = d;
        const double inv = fast_rcp(d);
        double cs[D];
#pragma unroll
        for(int i = 0; i < D; i++) cs[i] = a[i][s] * inv;
#pragma unroll
        for(int i = 0; i < D; i++)
#pragma unroll
            for(int j = 0; j < D; j++)
                if(i != s && j != s) a[i][j] -= cs[i] * a[s][j];
#pragma unroll
        for(int j = 0; j < D; j++)
            if(j != s) {
                a[s][j] *= inv;
                a[j][s] = cs[j];
            }
        a[s][s] = -inv;
    }
#pragma unroll
    for(int p = 0; p < D; p++)
#pragma unroll
        for(int q = 0; q < D; q++) Bout[p * D + q] = -a[p][q];
}

// publish the panel block of vertex v for the next step: P[p][x] = X(x, p), X(x, p) = TRANSPOSED ? a[p][x] : a[x][p]
template <int D, bool TRANSPOSED>
__device__ __forceinline__ void publish_panel(const double (&a)[D][D], double *Pb) {
#pragma unroll
    for(int p = 0; p < D; p++)
#pragma unroll
        for(int x = 0; x < D; x++) Pb[p * D + x] = TRANSPOSED ? a[p][x] : a[x][p];
}

// Shared-memory panels of one matrix in a block sweep: B x2 (inverted pivot block), P x2 (pivot panel), W (swept
// panel), piv (its scalar pivots, in sweep order), nsv: vertices swept (0: no such matrix).
struct SweepSet {
    double *B, *P, *W, *piv;
    int nsv;
};

// Sweeps the first nsv vertices of the symmetric matrix held in the blocks (active: vr < nsv): a <- -(A^-1) on the
// leading block. Pivot j is left in piv[j].
// Per vertex J, two phases with one barrier each:
//   1. the swept panel W_v = P_v B for every other vertex v (P_v = A_vJ and B = A_JJ^-1 were published during the
//      previous phase 2): one row of one W_v per thread of the CTA (G = 0), or two lanes per vertex of the group;
//   2. every block (I, L) off the pivot row / column: a -= W_I P_L^T (216 independent DFMAs, 16-byte operand
//      loads); blocks on the pivot row / column take W; the blocks of vertex J + 1 publish the next panel and
//      the thread of the next diagonal block inverts it in registers.
// G = 0 may sweep two independent matrices s0 and s1 in the same steps (s1.nsv > 0): the thread's block belongs to s1
// when own1, and phase 1 forms the W rows of both. Every element sees the same operations in the same order as in a
// sweep of its matrix alone; the step count is the larger nsv, the barriers are shared.
// Returns (uniformly) bit 0 / bit 1: a non-positive pivot in s0 / s1.
template <int D, int G>
__device__ __forceinline__ int block_sweep(double (&a)[D][D], const SweepSet &s0, const SweepSet &s1, bool own1, int vr, int vc,
                                           bool active, int nkmax) {
    constexpr int DD = D * D, PST = FastPad<D>::PST;
    constexpr int HS = (D % 2 == 0) ? 2 : 1; // lanes per vertex in phase 1 (nsv <= 16 vertices: otherwise one lane each)
    const int pstride = nkmax * PST;
    const int tid = Grp<G>::tid();
    constexpr int LW = G ? G : 32; // lanes of phase 1
    const SweepSet m = own1 ? s1 : s0; // the matrix of this thread's block
    const int nsv = m.nsv, nsteps = max(s0.nsv, s1.nsv);
    bool bad = false;
    if(active) {
        if(vc == 0 && vr > 0) publish_panel<D, false>(a, m.P + vr * PST);
        if(vr == 0 && vc == 0) invert_tile<D>(a, m.B, m.piv, bad);
    }
    Grp<G>::sync();
    const int hs = (HS * s0.nsv <= LW) ? HS : 1;
#pragma unroll 1
    for(int J = 0; J < nsteps; J++) {
        // ---- phase 1: W_v[q][x] = sum_p P_v[p][x] B[q][p] -----------------------------------------------------------
        if constexpr(G == 0) {
            // every thread of the CTA: one row q of one W_v, D independent chains summed over p in the same order as
            // the lane path below (bit-identical results). Row-major P_v rows and B rows: 16-byte loads and stores.
            // Rows of s0 first, then those of s1.
            const int n0 = J < s0.nsv ? s0.nsv * D : 0, n1 = J < s1.nsv ? s1.nsv * D : 0;
            for(int it = tid; it < n0 + n1; it += Grp<G>::nt()) {
                const bool second = it >= n0;
                const int i = second ? it - n0 : it, v = i / D, q = i % D;
                if(v == J) continue;
                const SweepSet &S = second ? s1 : s0;
                const double *Pv = S.P + (J & 1) * pstride + v * PST, *Bq = S.B + (J & 1) * DD + q * D;
                double w[D];
#pragma unroll
                for(int x = 0; x < D; x++) w[x] = 0;
#pragma unroll
                for(int p = 0; p < D; p++) {
                    const double b = Bq[p];
                    double px[D];
                    if constexpr(D % 2 == 0) { // all offsets are even numbers of doubles
#pragma unroll
                        for(int x = 0; x < D; x += 2) {
                            const double2 t = *reinterpret_cast<const double2 *>(Pv + p * D + x);
                            px[x] = t.x; px[x + 1] = t.y;
                        }
                    } else {
#pragma unroll
                        for(int x = 0; x < D; x++) px[x] = Pv[p * D + x];
                    }
#pragma unroll
                    for(int x = 0; x < D; x++) w[x] += px[x] * b;
                }
                double *Wq = S.W + v * PST + q * D;
                if constexpr(D % 2 == 0) {
#pragma unroll
                    for(int x = 0; x < D; x += 2) *reinterpret_cast<double2 *>(Wq + x) = make_double2(w[x], w[x + 1]);
                } else {
#pragma unroll
                    for(int x = 0; x < D; x++) Wq[x] = w[x];
                }
            }
        } else if(tid < LW) { // G > 0: s0 only
            const double *B = s0.B + (J & 1) * DD;
#pragma unroll 1
            for(int v0 = 0; v0 < s0.nsv; v0 += LW / hs) {
                const int v = v0 + tid / hs, h = tid % hs;
                if(v < s0.nsv && v != J) {
                    const int q0 = h * (D / hs), q1 = q0 + D / hs;
                    const double *Pv = s0.P + (J & 1) * pstride + v * PST;
                    double *Wv = s0.W + v * PST;
                    if(hs == HS) {
                        double bq[D / HS][D];
#pragma unroll
                        for(int q = 0; q < D / HS; q++)
#pragma unroll
                            for(int p = 0; p < D; p++) bq[q][p] = B[(q0 + q) * D + p];
#pragma unroll
                        for(int x = 0; x < D; x++) {
                            double px[D];
#pragma unroll
                            for(int p = 0; p < D; p++) px[p] = Pv[p * D + x];
#pragma unroll
                            for(int q = 0; q < D / HS; q++) {
                                double w = 0;
#pragma unroll
                                for(int p = 0; p < D; p++) w += px[p] * bq[q][p];
                                Wv[(q0 + q) * D + x] = w;
                            }
                        }
                    } else {
                        for(int q = q0; q < q1; q++)
                            for(int x = 0; x < D; x++) {
                                double w = 0;
#pragma unroll
                                for(int p = 0; p < D; p++) w += Pv[p * D + x] * B[q * D + p];
                                Wv[q * D + x] = w;
                            }
                    }
                }
            }
        }
        Grp<G>::sync();
        // ---- phase 2 ---------------------------------------------------------------------------------------------
        if(active && J < nsv && !(vr == J && vc == J)) {
            const double *Pc = m.P + (J & 1) * pstride;
            double *Pn = m.P + ((J + 1) & 1) * pstride;
            if(vc == J) { // block (I, J) <- W_I
                const double *Wb = m.W + vr * PST;
#pragma unroll
                for(int q = 0; q < D; q++)
#pragma unroll
                    for(int x = 0; x < D; x++) a[x][q] = Wb[q * D + x];
            } else if(vr == J) { // block (J, L) <- B A_JL = W_L^T
                const double *Wb = m.W + vc * PST;
#pragma unroll
                for(int q = 0; q < D; q++)
#pragma unroll
                    for(int x = 0; x < D; x++) a[q][x] = Wb[q * D + x];
            } else {
                const double *Wb = m.W + vr * PST, *Pb = Pc + vc * PST;
#pragma unroll
                for(int p = 0; p < D; p++) {
                    double w[D], q[D];
                    if constexpr(D % 2 == 0) { // 16-byte loads (all offsets are even numbers of doubles)
#pragma unroll
                        for(int r = 0; r < D; r += 2) {
                            const double2 t = *reinterpret_cast<const double2 *>(Wb + p * D + r);
                            w[r] = t.x; w[r + 1] = t.y;
                            const double2 u = *reinterpret_cast<const double2 *>(Pb + p * D + r);
                            q[r] = u.x; q[r + 1] = u.y;
                        }
                    } else {
#pragma unroll
                        for(int r = 0; r < D; r++) w[r] = Wb[p * D + r];
#pragma unroll
                        for(int c = 0; c < D; c++) q[c] = Pb[p * D + c];
                    }
#pragma unroll
                    for(int r = 0; r < D; r++)
#pragma unroll
                        for(int c = 0; c < D; c++) a[r][c] -= w[r] * q[c];
                }
            }
            if(J + 1 < nsv) {
                if(vc == J + 1) {
                    if(vr == J + 1) invert_tile<D>(a, m.B + ((J + 1) & 1) * DD, m.piv + D * (J + 1), bad);
                    else publish_panel<D, false>(a, Pn + vr * PST);
                } else if(vr == J + 1) publish_panel<D, true>(a, Pn + vc * PST);
            }
        }
        Grp<G>::sync();
    }
    const int bad0 = Grp<G>::any(bad && !own1) ? 1 : 0;
    return (s1.nsv > 0 && Grp<G>::any(bad && own1)) ? (bad0 | 2) : bad0;
}

// Cholesky of the diagonal block C_vv = -a held in registers. Lout: column-major D x D, strictly-lower entries of
// L and the RECIPROCALS of its diagonal; Cout: the block itself (column-major). Returns logdet C_vv.
template <int D>
__device__ __forceinline__ double chol_tile(const double (&a)[D][D], double *Lout, double *Cout, bool &ok) {
    double L[D][D];
    double lds = 0;
    ok = true;
#pragma unroll
    for(int c = 0; c < D; c++) {
        double d = -a[c][c];
#pragma unroll
        for(int p = 0; p < c; p++) d -= L[c][p] * L[c][p];
        if(!(d > 0)) { ok = false; d = 1.0; }
        lds += log(d);
        const double il = rsqrt(d);
        L[c][c] = il;
#pragma unroll
        for(int r = c + 1; r < D; r++) {
            double s = -a[r][c];
#pragma unroll
            for(int p = 0; p < c; p++) s -= L[r][p] * L[c][p];
            L[r][c] = s * il;
        }
    }
#pragma unroll
    for(int c = 0; c < D; c++)
#pragma unroll
        for(int r = 0; r < D; r++) {
            Lout[r + c * D] = (r >= c) ? L[r][c] : 0.0;
            Cout[r + c * D] = -a[r][c];
        }
    return lds;
}

// logdet (C_jj - C_ji C_ii^-1 C_ij), i < j: C_ji = -a (rows: components of j, columns: components of i) in
// registers, Li = chol_tile(C_ii), Cjj = the published diagonal block (pseudo_chow_liu.cpp:169-183)
template <int D>
__device__ __forceinline__ double schur_logdet_tile(const double (&a)[D][D], const double *Li, const double *Cjj) {
    double Y[D][D]; // Y = Li^-1 C_ij, D x D: row r (component of i), column c (component of j)
#pragma unroll
    for(int c = 0; c < D; c++) {
#pragma unroll
        for(int r = 0; r < D; r++) {
            double s = -a[c][r];
#pragma unroll
            for(int p = 0; p < r; p++) s -= Li[r + p * D] * Y[p][c];
            Y[r][c] = s * Li[r + r * D];
        }
    }
    double S[D][D];
#pragma unroll
    for(int c = 0; c < D; c++)
#pragma unroll
        for(int r = c; r < D; r++) {
            double s = Cjj[r + c * D];
#pragma unroll
            for(int p = 0; p < D; p++) s -= Y[p][r] * Y[p][c];
            S[r][c] = s;
        }
    double ld_sum = 0;
    double dinv[D];
#pragma unroll
    for(int c = 0; c < D; c++) {
        double d = S[c][c];
#pragma unroll
        for(int p = 0; p < c; p++) d -= S[c][p] * S[c][p] * dinv[p];
        ld_sum += log(d);
        dinv[c] = fast_rcp(d);
#pragma unroll
        for(int r = c + 1; r < D; r++) {
            double s = S[r][c];
#pragma unroll
            for(int p = 0; p < c; p++) s -= S[r][p] * S[c][p] * dinv[p];
            S[r][c] = s;
        }
    }
    return ld_sum;
}

// shared-memory plan of ONE blanket slot of fast_kernel (doubles; struct FastPlan in spg_plan.h), computed on the host.
// fused: the C and G sweeps run side by side (see fast_kernel S3), with a second panel set and a pivot array for C.
template <int D>
inline FastPlan fast_plan(int max_nv, int max_e, int max_rec_words, size_t smem_budget_bytes, bool fused) {
    constexpr int PS = PoseStride<D>::value;
    constexpr int JW = 2 * D * D, SW = 4 * D * D, PST = FastPad<D>::PST;
    FastPlan p;
    const int nk = max_nv > 1 ? max_nv - 1 : 1, kmax = D * nk, pairs = nk * (nk - 1) / 2;
    const int me = max_e < 1 ? 1 : max_e;
    p.NP = kmax;
    p.ntiles = nk * (nk + 1) / 2;
    int o = 0;
    p.off_pose = o;  o += max_nv * PS;
    p.off_small = o;
    // wt[pairs] heapw[pairs] heapab[pairs](int) tree[2 pairs + 2](int) uf[nk](int) ev[max_e](int) star[5 nk](int)
    // Lfac[nk D D] Cd[nk D D] logd[nk] cs[kmax] piv[kmax] red[34] misc[16](int)
    o += 2 * pairs + (pairs + 1) / 2 + (pairs + 1) + (nk + 2) / 2 + (me + 2) / 2 + (5 * nk + 2) / 2 + 2 * nk * D * D + nk + 2 * kmax + 34 + 8;
    o = (o + 1) & ~1;
    p.off_U = o;
    // union region.
    //   A (assembly, Schur): record | H00 x2 | H_k0 | Y | J, M of a chunk of edges
    //   B (Schur .. anchored sweep): the Lambda_t blocks [element][tile] | B x2 | P x2 | W   (block sweep panels)
    //     fused: ... | B2 x2 | P2 x2 | W2 | piv2[kmax]   (panels of the second matrix, pivots of the first)
    //   C (closed form): Jn | Sg | Tm | Bk
    const int rec = (max_rec_words + 1) & ~1;
    const int h0 = 2 * D * D + 2 * D * kmax;
    const int tb = (p.ntiles * D * D + 1) & ~1;
    const int set = 2 * D * D + 3 * nk * PST; // one panel set
    const int B = tb + set + (fused ? set + ((kmax + 1) & ~1) : 0);
    const int C = (nk > 1 ? nk - 1 : 1) * (2 * JW + SW + D * D);
    const int emin = me < 4 ? me : 4;
    int U = rec + h0 + emin * 2 * JW;
    if(B > U) U = B;
    if(C > U) U = C;
    // all edges in one assembly pass when that still leaves room for the resident CTAs the registers allow
    const int Ufull = rec + h0 + me * 2 * JW;
    if(Ufull > U && (size_t) (p.off_U + Ufull) * sizeof(double) <= smem_budget_bytes) U = Ufull;
    p.chunk = (U - rec - h0) / (2 * JW);
    if(p.chunk > me) p.chunk = me;
    if(p.chunk < 1) p.chunk = 1;
    p.off_h00 = p.off_U + rec;
    p.off_hk0 = p.off_h00 + 2 * D * D;
    p.off_y = p.off_hk0 + D * kmax;
    p.off_jm = p.off_y + D * kmax;
    p.off_B = p.off_U + tb;
    p.off_P = p.off_B + 2 * D * D;
    p.off_W = p.off_P + 2 * nk * PST;
    p.off_set2 = fused ? set : 0;
    p.total = (p.off_U + U + 1) & ~1;
    return p;
}
// threads that work on one blanket: one per block of the lower block triangle
__host__ __device__ inline int fast_tiles(int max_nv) {
    const int nk = max_nv > 1 ? max_nv - 1 : 1;
    return nk * (nk + 1) / 2;
}

#define SPG_FT(i)                                                                                    \
    do {                                                                                             \
        if(P.prof && tid == 0) {                                                                     \
            const long long t_now = clock64();                                                       \
            atomicAdd(&P.prof[i], (unsigned long long) (t_now - t_last));                            \
            t_last = t_now;                                                                          \
        }                                                                                            \
    } while(0)

// Phase barrier of the sub-warp-group kernels (G > 0). The warps of such a CTA work on different blankets and never
// exchange data, but the kernel is ~13 k instructions of mostly straight-line code against a 32 KB instruction cache:
// warps that drift apart each stream the whole kernel through the cache on their own (ncu, n = 8: 4.1 of 9.8 stall
// cycles per issue are `no_instruction`, 40 % of the instruction-cache requests miss). A CTA-wide barrier at every
// stage boundary keeps the warps of an SM inside the same few KB of code, so that a line is fetched once for all of
// them. barrier.sync (not .aligned): the groups of a warp may arrive from different places; every thread executes
// exactly FAST_PHASES barriers per blanket (stages it skips are made up for at the end of the iteration).
#define SPG_PHASE()                                                                                  \
    do {                                                                                             \
        if constexpr(G != 0) {                                                                       \
            if(phased) {                                                                             \
                asm volatile("barrier.sync 1;");                                                     \
                nb++;                                                                                \
            }                                                                                        \
        }                                                                                            \
    } while(0)
constexpr int FAST_PHASES = 9;
#define SPG_PHASE_CATCH_UP()                                                                         \
    do {                                                                                             \
        if constexpr(G != 0) {                                                                       \
            if(phased)                                                                               \
                for(; nb < FAST_PHASES; nb++) asm volatile("barrier.sync 1;");                       \
        }                                                                                            \
    } while(0)

// G: see Grp. MAXW: warps per CTA at most (G = 0: one blanket per CTA; G > 0: one blanket per group of G lanes).
template <int D, int G, int MAXW>
__global__ void __launch_bounds__(32 * MAXW, G ? 1 : (MAXW <= 4 ? 3 : (D == 6 ? 1 : 2))) fast_kernel(const KernelParams P) {
    extern __shared__ __align__(16) double fast_smem[];
    using GS = Grp<G>;
    constexpr int PS = PoseStride<D>::value;
    constexpr int PW = (D == 6) ? 7 : 3;
    constexpr int JW = D * 2 * D;
    constexpr int SW = 4 * D * D;
    constexpr int DD = D * D;
    const int tid = GS::tid(), NT = GS::nt();

    const FastPlan &pl = P.fast; // computed on the host (fast_plan): constant-bank loads
    double *smem = fast_smem + (size_t) GS::slot() * pl.total;
    const int NP = pl.NP;
    double *s_pose = smem + pl.off_pose;
    const int nkmax = P.max_nv > 1 ? P.max_nv - 1 : 1, kmaxb = pl.NP, pairs_max = nkmax * (nkmax - 1) / 2;
    const int me = P.max_e < 1 ? 1 : P.max_e;
    double *s_wt = smem + pl.off_small;
    double *s_heapw = s_wt + pairs_max;
    int *s_heapab = reinterpret_cast<int *>(s_heapw + pairs_max);
    int *s_tree = reinterpret_cast<int *>(s_heapw + pairs_max + (pairs_max + 1) / 2);
    int *s_uf = reinterpret_cast<int *>(s_heapw + pairs_max + (pairs_max + 1) / 2 + (pairs_max + 1));
    int *s_ev = reinterpret_cast<int *>(s_heapw + pairs_max + (pairs_max + 1) / 2 + (pairs_max + 1) + (nkmax + 2) / 2);
    int *s_star = reinterpret_cast<int *>(s_heapw + pairs_max + (pairs_max + 1) / 2 + (pairs_max + 1) + (nkmax + 2) / 2 + (me + 2) / 2);
    double *s_Lfac = s_heapw + pairs_max + (pairs_max + 1) / 2 + (pairs_max + 1) + (nkmax + 2) / 2 + (me + 2) / 2 + (5 * nkmax + 2) / 2;
    double *s_Cd = s_Lfac + nkmax * DD;
    double *s_logd = s_Cd + nkmax * DD;
    double *s_cs = s_logd + nkmax;
    double *s_piv = s_cs + kmaxb;
    double *s_red = s_piv + kmaxb;
    int *s_misc = reinterpret_cast<int *>(s_red + 34);
    double *U = smem + pl.off_U;
    uint64_t *s_rec = reinterpret_cast<uint64_t *>(U);
    double *s_h00 = smem + pl.off_h00; // 2 x D*D
    double *s_hk0 = smem + pl.off_hk0; // [D][NP]: H_k0, p-major
    double *s_y = smem + pl.off_y;     // [D][NP]: H_k0 H_00^-1
    double *JM = smem + pl.off_jm;     // per edge of a chunk: J = [Ji Jj], M = Omega J
    double *Tb = U;                    // Lambda_t blocks, [element][tile]
    double *s_B = smem + pl.off_B;
    double *s_P = smem + pl.off_P;
    double *s_W = smem + pl.off_W;
    const int tstride = pl.ntiles;

    const bool phased = G != 0 && blockDim.x > 32;
    for(int base = blockIdx.x * GS::slots(); base < P.n_list; base += gridDim.x * GS::slots()) {
        int nb = 0; // phase barriers executed in this iteration
        const int li = base + GS::slot();
        if(li >= P.n_list) { // no blanket for this group in the last iteration: it only keeps the barrier count
            SPG_PHASE_CATCH_UP();
            continue;
        }
        const int b = P.list ? P.list[li] : li;
        const uint64_t *grec = P.records + P.rec_off[b];
        uint64_t *gout = P.out + P.out_off[b];
        const int out_words = (int) (P.out_off[b + 1] - P.out_off[b]);
        const int32_t *gh = reinterpret_cast<const int32_t *>(grec);
        const int nv = gh[0], nrem = gh[1], ne = gh[2], rdim = gh[3], rec_words = gh[4];
        const int nk = nv - nrem, k = D * nk;

        GS::sync(); // the shared buffers of the previous blanket are dead
        SPG_PHASE(); // 1
        bool refuse = (rdim != D || nv > P.max_nv || ne > P.max_e || rec_words > P.max_rec_words || nrem != 1 || nk < 2 || ne < 1);
        for(int t = tid; t < out_words; t += NT) gout[t] = 0;
        long long t_last = clock64();
        if(!refuse) {
            for(int t = tid; t < rec_words; t += NT) s_rec[t] = grec[t];
            if(tid == 0) { s_misc[0] = 0; s_misc[3] = 0; }
        }
        GS::sync();
        const double *r_pose = reinterpret_cast<const double *>(s_rec + spgr_poses_off(nv));
        const int32_t *r_etab = reinterpret_cast<const int32_t *>(s_rec + spgr_edgetab_off(D, nv));
        if(!refuse) {
            // every edge a relative-pose edge between two different vertices? (anything else: blanket_kernel)
            int badedge = 0;
            for(int e = tid; e < ne; e += NT) {
                const int32_t *eh = reinterpret_cast<const int32_t *>(s_rec + r_etab[e]);
                const int32_t *vi = reinterpret_cast<const int32_t *>(s_rec + r_etab[e] + 2);
                badedge |= (eh[0] != SPG_EDGE_POSE) || (eh[1] != 2) || (vi[0] == vi[1]);
                s_ev[e] = pk(vi[0], vi[1]);
            }
            refuse = GS::any(badedge) != 0;
        }
        int n_out = 0;
        double out_kld = 0;
        int out_flags = 0;
        if(!refuse) {
            // ---- block of this thread: rows of kept vertex vr, columns of kept vertex vc <= vr ------------------
            // (fused sweeps: from S3 on, threads ntiles ... ntiles + gtiles - 1 hold the blocks of Lambda_rr, see S3 / S4)
            const int ntiles = nk * (nk + 1) / 2;
            bool has_tile = tid < ntiles;
            int vc = 0, vr = 0;
            if(has_tile) {
                int rem = tid;
                while(rem >= nk - vc) { rem -= nk - vc; vc++; }
                vr = vc + rem;
            }
            bool diag = has_tile && (vr == vc);
            double a[D][D];
#pragma unroll
            for(int r = 0; r < D; r++)
#pragma unroll
                for(int c = 0; c < D; c++) a[r][c] = 0.0;

            // ---- S0: poses; per kept vertex the edges to the removed vertex, in edge order (at most 4 parallel
            // edges, else blanket_kernel) ----------------------------------------------------------------------------
            for(int v = tid; v < nv; v += NT) {
                if constexpr(D == 6) se3_from_flat(r_pose + PW * v, s_pose + PS * v);
                else se2_from_flat(r_pose + PW * v, s_pose + PS * v);
            }
            int manystar = 0;
            for(int v = tid; v < nk; v += NT) {
                int cnt = 0;
                for(int e = 0; e < ne; e++) {
                    const int vab = s_ev[e], va = pk_a(vab), vb = pk_b(vab);
                    if((va == 0 && vb == v + 1) || (vb == 0 && va == v + 1)) {
                        if(cnt < 4) s_star[5 * v + 1 + cnt] = e;
                        cnt++;
                    }
                }
                s_star[5 * v] = cnt;
                manystar |= (cnt > 4);
            }
            for(int t = tid; t < DD + 2 * D * NP; t += NT) s_h00[DD + t] = 0.0; // second H00 buffer, H_k0, Y
            if(GS::any(manystar)) refuse = true;
            SPG_FT(0);
            SPG_PHASE(); // 2
            // ---- S1: assembly. Per chunk of edges (normally all of them): one thread per edge writes J = [Ji Jj] and
            // M = Omega J to shared memory, then every block gathers the edges of its vertex pair in edge order
            // (fixed summation order), and D (k + D) threads gather H_00 and H_k0 from the edges to the removed vertex.
            const int chunk = pl.chunk;
            for(int e0 = 0; e0 < ne && !refuse; e0 += chunk) {
                const int ce = min(chunk, ne - e0);
                for(int e = tid; e < ce; e += NT) {
                    const uint64_t *ew = s_rec + r_etab[e0 + e];
                    const int32_t *vi = reinterpret_cast<const int32_t *>(ew + 2);
                    const double *pm = reinterpret_cast<const double *>(ew + 3);
                    const double *Om = pm + PW;
                    double *J = JM + (size_t) e * 2 * JW;
                    double Z[PS];
                    if constexpr(D == 6) se3_from_flat(pm, Z);
                    else se2_from_flat(pm, Z);
                    edge_jacobians<D, G != 0>(Z, s_pose + PS * vi[0], s_pose + PS * vi[1], J);
                    if(e == 0) SPG_FT(8);
                    double om[D][D]; // Omega (symmetric), in registers for the 2 D columns of M = Omega J
#pragma unroll
                    for(int r = 0; r < D; r++)
#pragma unroll
                        for(int p2 = 0; p2 < D; p2++) om[r][p2] = Om[r + p2 * D];
#pragma unroll 1
                    for(int c = 0; c < 2 * D; c++) {
                        double jc[D];
#pragma unroll
                        for(int p2 = 0; p2 < D; p2++) jc[p2] = J[p2 + c * D];
#pragma unroll
                        for(int r = 0; r < D; r++) {
                            double sm = 0;
#pragma unroll
                            for(int p2 = 0; p2 < D; p2++) sm += om[r][p2] * jc[p2];
                            J[JW + r + c * D] = sm;
                        }
                    }
                }
                SPG_FT(9);
                GS::sync();
                SPG_FT(10);
                if(e0 == 0) SPG_PHASE(); // 3
                if(has_tile) {
                    const int lr = vr + 1, lc = vc + 1; // local vertex indices (the removed vertex is 0)
                    for(int e = 0; e < ce; e++) {
                        const int vab = s_ev[e0 + e];
                        const int va = pk_a(vab), vb = pk_b(vab);
                        int sr, sc; // side (0: Ji / first vertex, 1: Jj) of the row vertex and of the column vertex
                        if(va == lr) sr = 0; else if(vb == lr) sr = 1; else continue;
                        if(va == lc) sc = 0; else if(vb == lc) sc = 1; else continue;
                        const double *Jr = JM + (size_t) e * 2 * JW + sr * DD;
                        const double *Mc = JM + (size_t) e * 2 * JW + JW + sc * DD;
#pragma unroll
                        for(int p = 0; p < D; p++) {
                            double jr[D], mc[D];
#pragma unroll
                            for(int r = 0; r < D; r++) jr[r] = Jr[p + r * D];
#pragma unroll
                            for(int c = 0; c < D; c++) mc[c] = Mc[p + c * D];
#pragma unroll
                            for(int r = 0; r < D; r++)
#pragma unroll
                                for(int c = 0; c < D; c++) a[r][c] += jr[r] * mc[c];
                        }
                    }
                }
                SPG_FT(11);
                // H_k0: entry (i, p), i in [0, k): the edges between the removed vertex and kept vertex i / D
                for(int t = tid; t < k * D; t += NT) {
                    const int i = t % k, p = t / k, v = i / D, di = i % D;
                    const int cnt = s_star[5 * v];
                    double s = 0;
                    for(int q = 0; q < cnt; q++) {
                        const int e = s_star[5 * v + 1 + q] - e0;
                        if(e < 0 || e >= ce) continue;
                        const int sv = (pk_a(s_ev[e0 + e]) == 0) ? 1 : 0; // side of the kept vertex
                        const double *Jv = JM + (size_t) e * 2 * JW + (sv * D + di) * D;
                        const double *M0 = JM + (size_t) e * 2 * JW + JW + ((1 - sv) * D + p) * D;
#pragma unroll
                        for(int q2 = 0; q2 < D; q2++) s += Jv[q2] * M0[q2];
                    }
                    s_hk0[p * NP + i] += s;
                }
                // H_00: every edge of the removed vertex
                for(int t = tid; t < DD; t += NT) {
                    const int di = t % D, p = t / D;
                    double s = 0;
                    for(int e = 0; e < ce; e++) {
                        const int vab = s_ev[e0 + e];
                        int s0;
                        if(pk_a(vab) == 0) s0 = 0; else if(pk_b(vab) == 0) s0 = 1; else continue;
                        const double *J0 = JM + (size_t) e * 2 * JW + (s0 * D + di) * D;
                        const double *M0 = JM + (size_t) e * 2 * JW + JW + (s0 * D + p) * D;
#pragma unroll
                        for(int q2 = 0; q2 < D; q2++) s += J0[q2] * M0[q2];
                    }
                    s_h00[DD + di + p * D] += s;
                }
                GS::sync();
            }
            SPG_FT(1);
            SPG_PHASE(); // 4
            // ---- S2: Schur complement Lambda_t = H_kk - H_k0 H_00^-1 H_0k (vertex_remover.cpp:443-449) ---------
            // H_00^-1 by D symmetric Gauss-Jordan steps (a pivot <= 0 is LLT's failure)
            if(!refuse) {
                double *src = s_h00 + DD, *dst = s_h00;
                for(int s0 = 0; s0 < D; s0++) {
                    for(int t = tid; t < DD; t += NT) {
                        const int i = t % D, j = t / D;
                        const double d = src[s0 + s0 * D];
                        if(!(d > 0)) s_misc[0] = 1;
                        const double inv = fast_rcp(d), bis = src[i + s0 * D], bsj = src[s0 + j * D];
                        double v = src[i + j * D] - bis * bsj * inv;
                        if(j == s0) v = bis * inv;
                        if(i == s0) v = bsj * inv;
                        if(i == s0 && j == s0) v = -inv;
                        dst[t] = v;
                    }
                    GS::sync();
                    double *tmp = src; src = dst; dst = tmp;
                }
                const double *Hinv = src; // -H_00^-1
                for(int t = tid; t < k * D; t += NT) { // Y[p][i] = sum_q H_k0[q][i] * H_00^-1[q][p]
                    const int i = t % k, p = t / k;
                    double s = 0;
#pragma unroll
                    for(int q = 0; q < D; q++) s -= s_hk0[q * NP + i] * Hinv[q + p * D];
                    s_y[p * NP + i] = s;
                }
                GS::sync();
                if(s_misc[0]) refuse = true; // uniform (read after the barrier)
            }
            int bigdiag = 0;
            if(!refuse) {
                if(has_tile) {
#pragma unroll
                    for(int p = 0; p < D; p++) {
                        double yi[D], hl[D];
#pragma unroll
                        for(int r = 0; r < D; r++) yi[r] = s_y[p * NP + D * vr + r];
#pragma unroll
                        for(int c = 0; c < D; c++) hl[c] = s_hk0[p * NP + D * vc + c];
#pragma unroll
                        for(int r = 0; r < D; r++)
#pragma unroll
                            for(int c = 0; c < D; c++) a[r][c] -= yi[r] * hl[c];
                    }
                    if(diag) { // strict upper mirrored onto the strict lower triangle (:447-449); guard (ii) of S4
#pragma unroll
                        for(int r = 0; r < D; r++)
#pragma unroll
                            for(int c = 0; c < D; c++)
                                if(r > c) a[r][c] = a[c][r];
#pragma unroll
                        for(int r = 0; r < D; r++) bigdiag |= !(fabs(a[r][r]) < 1e8);
                    }
                }
                if(P.dbg_target && has_tile) {
                    double *g = P.dbg_target + P.dbg_target_off[b];
                    if(P.dbg_target_off[b + 1] - P.dbg_target_off[b] >= (int64_t) k * k) {
#pragma unroll
                        for(int r = 0; r < D; r++)
#pragma unroll
                            for(int c = 0; c < D; c++) {
                                g[(D * vr + r) + (size_t) (D * vc + c) * k] = a[r][c];
                                g[(D * vc + c) + (size_t) (D * vr + r) * k] = a[r][c];
                            }
                    }
                }
                GS::sync(); // Y, H_k0 and the record are dead: the union region now holds the Lambda_t blocks and the panels
                if(has_tile) {
#pragma unroll
                    for(int r = 0; r < D; r++)
#pragma unroll
                        for(int c = 0; c < D; c++) Tb[(r + c * D) * tstride + tid] = a[r][c];
                }
            }
            SPG_FT(2);
            SPG_PHASE(); // 5
            // ---- S3: Chow-Liu tree (pseudo_chow_liu.cpp:33-87) --------------------------------------------------
            // Fused (the host gave the CTA nkmax^2 threads and a second panel set): the anchored G = Lambda_rr^-1 of S4
            // is swept in the same block steps as C, on the threads past the C blocks. A failed G pivot is kept in
            // g_bad and refuses the blanket where the serial order meets it, after guard (ii).
            const bool fused = pl.off_set2 != 0 && nk > 2;
            const int gtiles = (nk - 1) * nk / 2;
            const bool g_own = fused && tid >= ntiles && tid < ntiles + gtiles;
            bool g_bad = false;
            if(!refuse) {
                if(nk == 2) {
                    n_out = 1;
                    if(tid == 0) s_tree[0] = pk(0, 1);
                } else {
                    n_out = nk - 1;
                    const int all = nk * (nk - 1) / 2;
                    // C = (Lambda_t + 1 I)^-1 (fillEdges, :185-190): symmetric sweep of the blocks
                    if(diag) {
#pragma unroll
                        for(int r = 0; r < D; r++) a[r][r] += 1.0;
                    }
                    SweepSet sc{s_B, s_P, s_W, s_piv, nk}, sg{nullptr, nullptr, nullptr, nullptr, 0};
                    if(fused) {
                        double *B2 = s_B + pl.off_set2;
                        sg = SweepSet{B2, B2 + 2 * DD, B2 + 2 * DD + 2 * nkmax * FastPad<D>::PST, s_piv, nk - 1};
                        sc.piv = sg.W + nkmax * FastPad<D>::PST; // C's pivots are not used after the sweep
                        GS::sync(); // the Lambda_t blocks are written
                        if(g_own) { // block (vr, vc) of the first nk - 1 vertices, loaded from the Lambda_t blocks
                            int rem = tid - ntiles;
                            while(rem >= nk - 1 - vc) { rem -= nk - 1 - vc; vc++; }
                            vr = vc + rem;
                            const int t = vc * nk - vc * (vc - 1) / 2 + (vr - vc);
#pragma unroll
                            for(int r = 0; r < D; r++)
#pragma unroll
                                for(int c = 0; c < D; c++) a[r][c] = Tb[(r + c * D) * tstride + t];
                        }
                    }
                    const int swept = block_sweep<D, G>(a, sc, sg, g_own, vr, vc, has_tile || g_own, nkmax);
                    if(swept & 1) refuse = true;
                    g_bad = (swept & 2) != 0;
                    if(!refuse) {
                        SPG_FT(3);
                        SPG_PHASE(); // 6
                        if(diag) {
                            bool ok;
                            s_logd[vr] = chol_tile<D>(a, s_Lfac + vr * DD, s_Cd + vr * DD, ok);
                            if(!ok) s_misc[0] = 1;
                        }
                        GS::sync();
                        // weight(i,j) = logdet C_jj - logdet (C_jj - C_ji C_ii^-1 C_ij)   (:169-183)
                        if(has_tile && !diag) {
                            const int i = vc, j = vr;
                            const int t = i * nk - (i * (i + 1)) / 2 + (j - i - 1);
                            s_wt[t] = s_logd[j] - schur_logdet_tile<D>(a, s_Lfac + i * DD, s_Cd + j * DD);
                        }
                        GS::sync();
                        if(s_misc[0]) refuse = true;
                    }
                    if(!refuse) {
                        if(P.dbg_weights) {
                            double *g = P.dbg_weights + P.dbg_weights_off[b];
                            const int cap = (int) (P.dbg_weights_off[b + 1] - P.dbg_weights_off[b]);
                            if(P.flags & SPG_OPT_DBG_WEIGHTS_IN) {
                                for(int t = tid; t < all && t < cap; t += NT) s_wt[t] = g[t];
                                GS::sync();
                            } else {
                                for(int t = tid; t < cap; t += NT) g[t] = t < all ? s_wt[t] : 0.0;
                            }
                        }
                        SPG_FT(4);
                        SPG_PHASE(); // 7
                        // doKruskal (:253-289): same scheme as blanket_kernel — parallel ranking, or the replay of
                        // libstdc++'s heap when two weights are exactly equal
                        int *s_sorted = s_tree + all;
                        for(int t = tid; t < all; t += NT) {
                            const double wt = s_wt[t];
                            int rank = 0, tie = (wt != wt);
                            for(int u = 0; u < all; u++) {
                                const double wu = s_wt[u];
                                rank += (wu > wt);
                                tie |= (u != t) && (wu == wt);
                            }
                            if(tie) s_misc[3] = 1;
                            else {
                                int i = 0, rem = t;
                                while(rem >= nk - 1 - i) { rem -= nk - 1 - i; i++; }
                                s_sorted[rank] = pk(i, i + 1 + rem);
                            }
                        }
                        GS::sync();
                        if(s_misc[3]) out_flags |= 128;
                        if(tid == 0) {
                            for(int v = 0; v < nk; v++) s_uf[v] = v;
                            int nacc = 0;
                            if(!s_misc[3]) {
                                for(int q = 0; q < all && nacc < nk - 1; q++) {
                                    const int ab = s_sorted[q];
                                    int ra = pk_a(ab), rbb = pk_b(ab);
                                    while(s_uf[ra] != ra) ra = s_uf[ra];
                                    while(s_uf[rbb] != rbb) rbb = s_uf[rbb];
                                    if(ra != rbb) {
                                        s_uf[rbb] = ra;
                                        s_tree[nacc++] = ab;
                                    }
                                }
                            } else {
                                HeapView hp{s_heapw, s_heapab, 0};
                                int t = 0;
                                for(int i = 0; i < nk - 1; i++)
                                    for(int j = i + 1; j < nk; j++, t++) hp.push(s_wt[t], pk(i, j));
                                while(hp.len > 0 && nacc < nk - 1) {
                                    double w; int ab;
                                    hp.pop(w, ab);
                                    int ra = pk_a(ab), rbb = pk_b(ab);
                                    while(s_uf[ra] != ra) ra = s_uf[ra];
                                    while(s_uf[rbb] != rbb) rbb = s_uf[rbb];
                                    if(ra != rbb) {
                                        s_uf[rbb] = ra;
                                        s_tree[nacc++] = ab;
                                    }
                                }
                            }
                        }
                        GS::sync();
                    }
                }
            }
            SPG_FT(5);
            SPG_PHASE(); // 8
            // ---- S4: gauge shortcut + closed form (see blanket_kernel for the argument) --------------------------
            const int kk = k - D;
            double glog = 0;
            if(!refuse) {
                // guard (ii): every diagonal entry of Lambda_t below 1e8
                if(GS::any(bigdiag)) refuse = true;
            }
            if(!refuse) {
                // G = Lambda_rr^-1 (last kept vertex anchored): the first nk - 1 vertices swept
                if(fused) {
                    // swept in S3. The blocks of G are the g_own threads'; the C threads of the anchored vertex's row
                    // hold zero blocks for the Sigma scatter, as the serial order below loads them
                    if(g_bad) refuse = true;
                    if(!g_own) {
#pragma unroll
                        for(int r = 0; r < D; r++)
#pragma unroll
                            for(int c = 0; c < D; c++) a[r][c] = 0.0;
                    }
                    has_tile = g_own || (has_tile && vr == nk - 1);
                    diag = has_tile && vr == vc;
                } else {
                    const bool act = has_tile && vr < nk - 1;
                    if(has_tile) {
#pragma unroll
                        for(int r = 0; r < D; r++)
#pragma unroll
                            for(int c = 0; c < D; c++) a[r][c] = act ? Tb[(r + c * D) * tstride + tid] : 0.0;
                    }
                    const SweepSet sg{s_B, s_P, s_W, s_piv, nk - 1}, none{nullptr, nullptr, nullptr, nullptr, 0};
                    if(block_sweep<D, G>(a, sg, none, false, vr, vc, act, nkmax)) refuse = true;
                }
                const bool act = has_tile && vr < nk - 1;
                if(!refuse) {
                    // guard (i): ||G||_F <= 1e5; log-determinant of Lambda_rr from the pivots
                    double fp = 0;
                    if(act) {
                        const double w = diag ? 1.0 : 2.0;
#pragma unroll
                        for(int r = 0; r < D; r++)
#pragma unroll
                            for(int c = 0; c < D; c++) fp += w * a[r][c] * a[r][c];
                    }
                    const double frob2 = GS::sum(fp, s_red);
                    if(!(frob2 <= 1e10)) refuse = true;
                    for(int t = tid; t < kk; t += NT) glog += log(s_piv[t]);
                }
            }
            SPG_FT(6);
            SPG_PHASE(); // 9
            if(!refuse) {
                // new-edge Jacobians at zero error (vertex_remover.cpp:466-498), Sigma blocks from G, X_e = (J Sigma J^T)^-1
                GS::sync();                               // the Lambda_t blocks and the panels are dead
                double *Jn = U;                           // n_out * JW
                double *Sg = Jn + (size_t) n_out * JW;    // n_out * SW
                double *Tm = Sg + (size_t) n_out * SW;    // n_out * JW
                double *Bk = Tm + (size_t) n_out * JW;    // n_out * D*D
                double *Bk2 = Sg;                         // ping-pong partner of Bk once Sg is consumed
                const int slot = 1 + PW + DD;
                for(int e = tid; e < n_out; e += NT) {
                    const int ea = pk_a(s_tree[e]), eb = pk_b(s_tree[e]);
                    const double *Xa = s_pose + PS * (1 + ea), *Xb = s_pose + PS * (1 + eb);
                    double Z[PS], Ti[PS];
                    if constexpr(D == 6) { se3_inverse(Xa, Ti); se3_compose(Ti, Xb, Z); }
                    else { se2_inverse(Xa, Ti); se2_compose(Ti, Xb, Z); }
                    edge_jacobians_zero_error<D>(Z, Xa, Xb, Jn + (size_t) e * JW);
                    uint64_t *sl = gout + SPG_OUT_HEADER_WORDS + (size_t) e * slot;
                    int32_t *si = reinterpret_cast<int32_t *>(sl);
                    si[0] = ea; si[1] = eb;
                    double *sm = reinterpret_cast<double *>(sl + 1);
                    if constexpr(D == 6) se3_to_flat<G != 0>(Z, sm);
                    else { sm[0] = Z[0]; sm[1] = Z[1]; sm[2] = Z[2]; }
                }
                // Sigma_e = [[G_aa G_ab] [G_ba G_bb]] scattered from the registers (G = -a; zero rows / columns for the
                // anchored vertex: its blocks were loaded as zeros)
                if(has_tile) {
                    for(int e = 0; e < n_out; e++) {
                        const int ea = pk_a(s_tree[e]), eb = pk_b(s_tree[e]);
                        double *S2 = Sg + (size_t) e * SW;
                        if(diag) {
                            if(vr == ea || vr == eb) {
                                const int o = (vr == ea) ? 0 : D;
#pragma unroll
                                for(int r = 0; r < D; r++)
#pragma unroll
                                    for(int c = 0; c < D; c++) S2[(o + r) + (o + c) * 2 * D] = (r >= c) ? -a[r][c] : -a[c][r];
                            }
                        } else if(vc == ea && vr == eb) {
#pragma unroll
                            for(int r = 0; r < D; r++)
#pragma unroll
                                for(int c = 0; c < D; c++) {
                                    S2[(D + r) + c * 2 * D] = -a[r][c];
                                    S2[c + (D + r) * 2 * D] = -a[r][c];
                                }
                        }
                    }
                }
                GS::sync();
                for(int t = tid; t < n_out * JW; t += NT) { // Tm = J Sigma_e
                    const int e = t / JW, q = t % JW, rr = q % D, j = q / D;
                    const double *J = Jn + (size_t) e * JW;
                    const double *S2 = Sg + (size_t) e * SW;
                    double acc = 0;
#pragma unroll
                    for(int i = 0; i < 2 * D; i++) acc += J[rr + i * D] * S2[i + j * 2 * D];
                    Tm[t] = acc;
                }
                GS::sync();
                for(int t = tid; t < n_out * DD; t += NT) { // block = Tm J^T, symmetrised (logdet_function.cpp:249-270)
                    const int e = t / DD, q = t % DD, rr = q % D, cc = q / D;
                    if(rr >= cc) {
                        const double *J = Jn + (size_t) e * JW;
                        const double *Te = Tm + (size_t) e * JW;
                        double s1 = 0, s2 = 0;
#pragma unroll
                        for(int j = 0; j < 2 * D; j++) {
                            s1 += Te[rr + j * D] * J[cc + j * D];
                            s2 += Te[cc + j * D] * J[rr + j * D];
                        }
                        const double v = 0.5 * (s1 + s2);
                        Bk[(size_t) e * DD + rr + cc * D] = v;
                        Bk[(size_t) e * DD + cc + rr * D] = v;
                    }
                }
                GS::sync();
                double *src = Bk, *dst = Bk2;
                for(int s0 = 0; s0 < D; s0++) { // X_e = block^-1 (:273-274), all blocks together, D Gauss-Jordan steps
                    for(int t = tid; t < n_out * DD; t += NT) {
                        const int e = t / DD, q = t % DD, i = q % D, j = q / D;
                        const double *B = src + (size_t) e * DD;
                        const double d = B[s0 + s0 * D];
                        if(!(d > 0)) s_misc[0] = 1;
                        if(i == s0 && j == s0) s_cs[e * D + s0] = d;
                        const double inv = fast_rcp(d), bis = B[i + s0 * D], bsj = B[s0 + j * D];
                        double v = B[i + j * D] - bis * bsj * inv;
                        if(j == s0) v = bis * inv;
                        if(i == s0) v = bsj * inv;
                        if(i == s0 && j == s0) v = -inv;
                        dst[t] = v;
                    }
                    GS::sync();
                    double *tmp = src; src = dst; dst = tmp;
                }
                if(s_misc[0]) refuse = true;
                if(!refuse) {
                    for(int t = tid; t < n_out * DD; t += NT) {
                        const int e = t / DD, q = t % DD;
                        double *sx = reinterpret_cast<double *>(gout + SPG_OUT_HEADER_WORDS + (size_t) e * slot + 1 + PW);
                        sx[q] = -src[t];
                    }
                    // projected KLD at the closed form = 1/2 [logdet Lambda_rr - sum_e logdet X_e] (see blanket_kernel)
                    double lp = glog;
                    for(int t = tid; t < n_out * D; t += NT) lp += log(s_cs[t]);
                    out_kld = 0.5 * GS::sum(lp, s_red);
                }
            }
            SPG_FT(7);
        }
        GS::sync();
        SPG_PHASE_CATCH_UP(); // stages this blanket skipped
        if(tid == 0) {
            int32_t *oh = reinterpret_cast<int32_t *>(gout);
            if(refuse) {
                oh[0] = SPG_BLANKET_UNSUPPORTED; // overwritten by blanket_kernel, which re-runs the blanket
                const int pos = atomicAdd(P.retry_count, 1);
                P.retry_list[pos] = b;
            } else {
                oh[0] = SPG_BLANKET_OK;
                oh[1] = n_out;
                oh[2] = 0;
                oh[3] = out_flags;
                reinterpret_cast<double *>(gout)[2] = out_kld;
            }
        }
    }
}

} // namespace spg
