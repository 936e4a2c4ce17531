// The step GTSAM performs after evaluateError, for an IMU-only chain, entirely on the device (SURVEY.md 8f rank 1):
//   k_factor_whiten   A = R_w [H1 H2], b = -R_w e  with the factor's noise model noiseModel::Gaussian::Covariance(P_meas)
//                     (gtsam/ImuFactorCPIv1.h:82, ImuFactorCPIv2.h:86): R_w = upper Cholesky factor of P_meas^-1, R_w^T R_w = P_meas^-1
//   k_chain_assemble  scatter-add of the per-factor information blocks into the block-tridiagonal normal equations of the chain
//                     x_0 - x_1 - ... - x_n  (what BatchFixedLagSmoother::update assembles, solvers/GraphSolver.cpp:202-203)
//   block cyclic reduction: a Cholesky-based solve of that SPD block-tridiagonal system (15x15 blocks) in log2(n) parallel levels
//                     instead of a 5 000-step sequential block recurrence: odd nodes are eliminated (one warp per node: Cholesky of the
//                     diagonal block + 31 forward substitutions), even nodes receive the Schur complements (one warp per node).
//   selected inversion: the same forward sweep without right-hand side, then from the root down, one warp per odd node, the diagonal and
//                     first off-diagonal 15x15 blocks of A^-1 (marginal covariances of every keyframe and of adjacent pairs, what GTSAM's
//                     Marginals::marginalCovariance / jointMarginalCovariance return) from the Cholesky factors and Lc^-1 E products the
//                     sweep left in the workspace: no dense inverse, 3 ceil(log2 n) + 1 launches.
// GTSAM is not part of the reference tree (bitbucket gtborg/gtsam @ c21186c): PARITY UNPINNED -- validated against dense / banded
// CPU solves of the same system (tests/test_gpu_parity.py) and, for the marginals, dense inverses and the forward-propagated covariance of
// the chain (tests/test_chain_marginals.py).
#include "cpi_common.cuh"
#include "cpi_kernels.h"

namespace cpi {

// ---- warp-level 15x15 helpers (matrix in shared memory, row-major with pitch 16) ---------------------------------------------------
// in-place lower Cholesky; a non-positive pivot gives NaN (GTSAM throws there)
CPI_DEV void warp_chol15(double* L, int lane) {
    for (int k = 0; k < 15; k++) {
        const double d = sqrt(L[k * 16 + k]);
        __syncwarp();
        if (lane == 0) L[k * 16 + k] = d;
        if (lane > k && lane < 15) L[lane * 16 + k] = L[lane * 16 + k] / d;
        __syncwarp();
        for (int t = lane; t < 120; t += 32) {
            int i = 0, acc = 0;
            while (acc + i + 1 <= t) { acc += i + 1; i++; }      // t -> (i, j) in the lower triangle incl. diagonal
            const int j = t - acc;
            if (j > k && i > k) L[i * 16 + j] -= L[i * 16 + k] * L[j * 16 + k];
        }
        __syncwarp();
    }
}
// y = L^-1 b  for a per-lane right-hand side held in registers (b -> y in place)
CPI_DEV void fwd15(const double* L, double* y) {
#pragma unroll
    for (int i = 0; i < 15; i++) {
        double t = y[i];
#pragma unroll
        for (int k = 0; k < i; k++) t = fma(-L[i * 16 + k], y[k], t);
        y[i] = t / L[i * 16 + i];
    }
}
// x = L^-T r : lane k (< 15) passes r_k and receives x_k; column-oriented backward substitution with shuffles
CPI_DEV double warp_bwd15(const double* L, double r, int lane) {
    double x = 0.0;
    for (int k = 14; k >= 0; k--) {
        const double xk = __shfl_sync(0xffffffffu, r, k) / L[k * 16 + k];
        if (lane == k) x = xk;
        if (lane < k) r = fma(-L[k * 16 + lane], xk, r);          // (L^T)[lane, k] = L[k, lane]
    }
    return x;
}

// x = L^-T y  for a per-lane right-hand side held in registers (y -> x in place)
CPI_DEV void bwd15(const double* L, double* y) {
#pragma unroll
    for (int i = 14; i >= 0; i--) {
        double t = y[i];
#pragma unroll
        for (int k = i + 1; k < 15; k++) t = fma(-L[k * 16 + i], y[k], t);
        y[i] = t / L[i * 16 + i];
    }
}
// M = L^-1 into shared memory (column-major; lane c < 15 forms column c); ends with __syncwarp
CPI_DEV void warp_inv_lower15(const double* L, double* M, int lane) {
    if (lane < 15) {
        double y[15];
#pragma unroll
        for (int i = 0; i < 15; i++) y[i] = (i == lane) ? 1.0 : 0.0;
        fwd15(L, y);
#pragma unroll
        for (int i = 0; i < 15; i++) M[i + 15 * lane] = y[i];
    }
    __syncwarp();
}
// (L L^T)^-1 [a, b] = (M^T M)[a, b] with M = L^-1: entries (a, b) and (b, a) sum the same products in the same order, so the result is
// exactly symmetric
CPI_DEV double inv_entry15(const double* M, int a, int b) {
    double s = 0.0;
    for (int k = a > b ? a : b; k < 15; k++) s = fma(M[k + 15 * a], M[k + 15 * b], s);
    return s;
}

// ---- explicitly whitened Jacobian form --------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) k_factor_whiten(int64_t n, int rd, const double* records, const double* e, const double* H1, const double* H2,
                                                       double* A1, double* A2, double* bw) {
    __shared__ double sL[4][15 * 16], sM[4][15 * 16], sR[4][15 * 16];
    const int wib = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t f = (int64_t)blockIdx.x * 4 + wib;
    if (f >= n) return;
    double *L = sL[wib], *M = sM[wib], *R = sR[wib];
    const double* P = records + f * (int64_t)rd + CPI_REC_P;
    for (int k = lane; k < 225; k += 32) { const int r = k % 15, c = k / 15; if (r >= c) L[r * 16 + c] = __ldg(P + k); }
    __syncwarp();
    warp_chol15(L, lane);                                          // P = L L^T
    // M = L^-1 (lane c: column c of the inverse), then information = M^T M
    if (lane < 15) {
        double y[15];
#pragma unroll
        for (int i = 0; i < 15; i++) y[i] = (i == lane) ? 1.0 : 0.0;
        fwd15(L, y);
#pragma unroll
        for (int i = 0; i < 15; i++) M[i * 16 + lane] = y[i];
    }
    __syncwarp();
    for (int t = lane; t < 225; t += 32) {                         // lower triangle of P^-1 = M^T M into R (to be factored in place)
        const int i = t / 15, j = t % 15;
        if (j <= i) {
            double s = 0.0;
            for (int k = i; k < 15; k++) s = fma(M[k * 16 + i], M[k * 16 + j], s);     // M is lower triangular: rows >= max(i, j)
            R[i * 16 + j] = s;
        }
    }
    __syncwarp();
    warp_chol15(R, lane);                                          // P^-1 = C C^T  ->  R_w = C^T (upper), R_w^T R_w = P^-1
    // A = R_w H:  (R_w H)[i, c] = sum_{k >= i} C[k, i] H[k, c];  lanes 0..14 -> columns of H1, 15..29 -> H2, 30 -> -e
    if (lane < 31) {
        const double* src = lane < 15 ? H1 + f * 225 + 15 * lane : (lane < 30 ? H2 + f * 225 + 15 * (lane - 15) : e + f * 15);
        double h[15];
#pragma unroll
        for (int i = 0; i < 15; i++) h[i] = __ldg(src + i);
        double* dst = lane < 15 ? A1 + f * 225 + 15 * lane : (lane < 30 ? A2 + f * 225 + 15 * (lane - 15) : bw + f * 15);
        const double sgn = lane < 30 ? 1.0 : -1.0;
#pragma unroll
        for (int i = 0; i < 15; i++) {
            double s = 0.0;
#pragma unroll
            for (int k = i; k < 15; k++) s = fma(R[k * 16 + i], h[k], s);
            dst[i] = sgn * s;
        }
    }
}

// ---- chain assembly ---------------------------------------------------------------------------------------------------------------
// Factor f links states f and f+1:  D[k] = G22[k-1] + G11[k] (+ prior on x_0) + damping,  E[k] = G12[k] (block (k, k+1)),  rhs[k] = g2[k-1] + g1[k].
// Damping as in GTSAM's LevenbergMarquardtParams: lambda I, or with diagonalDamping lambda * clamp(diag, minDiagonal 1e-6, maxDiagonal 1e32).
__global__ void k_chain_assemble(int64_t nf, const double* G11, const double* G12, const double* G22, const double* g1, const double* g2, double lambda,
                                 int diagonal_damping, const double* prior_info, const double* prior_rhs, double* D, double* E, double* rhs) {
    const int64_t k = blockIdx.x;                                  // state index 0..nf
    for (int t = threadIdx.x; t < 225; t += blockDim.x) {
        double d = 0.0;
        if (k > 0) d += G22[(k - 1) * 225 + t];
        if (k < nf) { d += G11[k * 225 + t]; E[k * 225 + t] = G12[k * 225 + t]; }
        if (k == 0 && prior_info) d += prior_info[t];
        if (t % 16 == 0) d += diagonal_damping ? lambda * fmin(fmax(d, 1e-6), 1e32) : lambda;     // t = r + 15 c: diagonal when r == c  <=>  t % 16 == 0
        D[k * 225 + t] = d;
    }
    for (int t = threadIdx.x; t < 15; t += blockDim.x) {
        double v = 0.0;
        if (k > 0) v += g2[(k - 1) * 15 + t];
        if (k < nf) v += g1[k * 15 + t];
        if (k == 0 && prior_rhs) v += prior_rhs[t];
        rhs[k * 15 + t] = v;
    }
}

// ---- block cyclic reduction ---------------------------------------------------------------------------------------------------------
// Level with m nodes: row i reads  E[i-1]^T x_{i-1} + D[i] x_i + E[i] x_{i+1} = b[i].
// Odd node i = 2t+1:  D_i = Lc Lc^T,  Za = Lc^-1 E[i-1]^T,  Zb = Lc^-1 E[i] (if i+1 < m),  zb = Lc^-1 b_i      (kept for the back-substitution)
// b = NULL (the marginals need no right-hand side) skips zb.
__global__ void __launch_bounds__(128) k_bcr_eliminate(int64_t m, const double* D, const double* E, const double* b, double* Lc, double* Za, double* Zb, double* zb) {
    __shared__ double sL[4][15 * 16];
    const int wib = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t t = (int64_t)blockIdx.x * 4 + wib;
    const int64_t i = 2 * t + 1;
    if (i >= m) return;
    double* L = sL[wib];
    for (int k = lane; k < 225; k += 32) { const int r = k % 15, c = k / 15; if (r >= c) L[r * 16 + c] = D[i * 225 + k]; }
    __syncwarp();
    warp_chol15(L, lane);
    for (int k = lane; k < 225; k += 32) { const int r = k % 15, c = k / 15; Lc[t * 225 + k] = (r >= c) ? L[r * 16 + c] : 0.0; }
    const bool has_right = i + 1 < m;
    if (lane < 30 || (lane == 30 && b)) {
        double y[15];
        if (lane < 15) {
#pragma unroll
            for (int r = 0; r < 15; r++) y[r] = E[(i - 1) * 225 + lane + 15 * r];          // column `lane` of E[i-1]^T = row `lane` of E[i-1]
        } else if (lane < 30) {
#pragma unroll
            for (int r = 0; r < 15; r++) y[r] = has_right ? E[i * 225 + r + 15 * (lane - 15)] : 0.0;
        } else {
#pragma unroll
            for (int r = 0; r < 15; r++) y[r] = b[i * 15 + r];
        }
        fwd15(L, y);
        double* dst = lane < 15 ? Za + t * 225 + 15 * lane : (lane < 30 ? Zb + t * 225 + 15 * (lane - 15) : zb + t * 15);
#pragma unroll
        for (int r = 0; r < 15; r++) dst[r] = y[r];
    }
}

// Even node j = 2u -> node u of the next level:
//   D' = D_j - Zb_{j-1}^T Zb_{j-1} - Za_{j+1}^T Za_{j+1},   b' = b_j - Zb_{j-1}^T zb_{j-1} - Za_{j+1}^T zb_{j+1},   E' = -Za_{j+1}^T Zb_{j+1}  (couples x_j and x_{j+2})
// b = NULL skips b'.
__global__ void __launch_bounds__(128) k_bcr_reduce(int64_t m, const double* D, const double* b, const double* Za, const double* Zb, const double* zb,
                                                    double* Dn, double* En, double* bn) {
    __shared__ double sZ[4][4][225 + 15];      // [warp][ZbL | ZaR | ZbR | (zbL, zbR)]
    const int wib = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t u = (int64_t)blockIdx.x * 4 + wib;
    const int64_t j = 2 * u;
    if (j >= m) return;
    const bool hasL = j >= 1, hasR = j + 1 < m, hasRR = j + 2 < m;
    const int64_t tl = (j - 2) / 2, tr = j / 2;                     // odd-node slots of j-1 and j+1
    double *ZbL = sZ[wib][0], *ZaR = sZ[wib][1], *ZbR = sZ[wib][2], *zz = sZ[wib][3];
    for (int k = lane; k < 225; k += 32) {
        ZbL[k] = hasL ? Zb[tl * 225 + k] : 0.0;
        ZaR[k] = hasR ? Za[tr * 225 + k] : 0.0;
        ZbR[k] = hasRR ? Zb[tr * 225 + k] : 0.0;
    }
    if (lane < 15 && b) { zz[lane] = hasL ? zb[tl * 15 + lane] : 0.0; zz[15 + lane] = hasR ? zb[tr * 15 + lane] : 0.0; }
    __syncwarp();
    for (int k = lane; k < 225; k += 32) {
        const int r = k % 15, c = k / 15;                          // column-major 15x15; Z matrices are column-major: Z[q + 15 col]
        double d = D[j * 225 + k], en = 0.0;
#pragma unroll
        for (int q = 0; q < 15; q++) {
            d = fma(-ZbL[q + 15 * r], ZbL[q + 15 * c], d);
            d = fma(-ZaR[q + 15 * r], ZaR[q + 15 * c], d);
            en = fma(-ZaR[q + 15 * r], ZbR[q + 15 * c], en);
        }
        Dn[u * 225 + k] = d;
        if (hasRR) En[u * 225 + k] = en;
    }
    if (lane < 15 && b) {
        double v = b[j * 15 + lane];
#pragma unroll
        for (int q = 0; q < 15; q++) { v = fma(-ZbL[q + 15 * lane], zz[q], v); v = fma(-ZaR[q + 15 * lane], zz[15 + q], v); }
        bn[u * 15 + lane] = v;
    }
}

// last level (one node): x = D^-1 b
__global__ void k_bcr_root(const double* D, const double* b, double* x, int64_t stride) {
    __shared__ double L[15 * 16];
    const int lane = threadIdx.x;
    for (int k = lane; k < 225; k += 32) { const int r = k % 15, c = k / 15; if (r >= c) L[r * 16 + c] = D[k]; }
    __syncwarp();
    warp_chol15(L, lane);
    double y[15];
#pragma unroll
    for (int r = 0; r < 15; r++) y[r] = b[r];
    fwd15(L, y);                                                   // every lane redundantly (15 x 15 / 2 fma)
    double r = 0.0;
#pragma unroll
    for (int q = 0; q < 15; q++) if (lane == q) r = y[q];
    const double xv = warp_bwd15(L, r, lane);
    if (lane < 15) x[lane] = xv;
    (void)stride;
}

// odd node i = 2t+1 of a level whose nodes sit at original indices i * stride:  Lc^T x_i = zb - Za x_{i-1} - Zb x_{i+1}
__global__ void __launch_bounds__(128) k_bcr_backsub(int64_t m, int64_t stride, const double* Lc, const double* Za, const double* Zb, const double* zb, double* x) {
    __shared__ double sL[4][15 * 16];
    const int wib = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t t = (int64_t)blockIdx.x * 4 + wib;
    const int64_t i = 2 * t + 1;
    if (i >= m) return;
    double* L = sL[wib];
    for (int k = lane; k < 225; k += 32) { const int r = k % 15, c = k / 15; if (r >= c) L[r * 16 + c] = Lc[t * 225 + k]; }
    __syncwarp();
    const bool has_right = i + 1 < m;
    double r = 0.0;
    if (lane < 15) {
        r = zb[t * 15 + lane];
        const double* xl = x + (i - 1) * stride * 15;
        const double* xr = x + (i + 1) * stride * 15;
#pragma unroll
        for (int q = 0; q < 15; q++) {
            r = fma(-Za[t * 225 + lane + 15 * q], xl[q], r);
            if (has_right) r = fma(-Zb[t * 225 + lane + 15 * q], xr[q], r);
        }
    }
    const double xv = warp_bwd15(L, r, lane);
    if (lane < 15) x[i * stride * 15 + lane] = xv;
}

// ---- selected inversion: diagonal and first off-diagonal blocks of Sigma = A^-1 --------------------------------------------------------
// Same forward sweep (without right-hand side), then level by level from the root down.  The coarse level's Sigma is the Sigma of the
// finer level restricted to its even nodes (the inverse of a Schur complement is a block of the inverse).

// last level (one node): Sigma = D^-1
__global__ void k_bcr_root_inv(const double* D, double* S) {
    __shared__ double L[15 * 16], M[225];
    const int lane = threadIdx.x;
    for (int k = lane; k < 225; k += 32) { const int r = k % 15, c = k / 15; if (r >= c) L[r * 16 + c] = D[k]; }
    __syncwarp();
    warp_chol15(L, lane);
    warp_inv_lower15(L, M, lane);
    for (int k = lane; k < 225; k += 32) S[k] = inv_entry15(M, k % 15, k / 15);
}

// Odd node i = 2t+1 of a level whose nodes sit at original indices i * stride.  Its neighbours l = i-1, r = i+1 are the coarse nodes t, t+1,
// whose blocks Sigma_ll, Sigma_rr (in S) and Sigma_lr (the coarse off-diagonal block t, in Sc) the level above produced.  With
// W_l = Lc^-T Za = D_i^-1 E[i-1]^T and W_r = Lc^-T Zb = D_i^-1 E[i] (zero without a right neighbour):
//   Sigma_il = -(W_l Sigma_ll + W_r Sigma_lr^T),   Sigma_ir = -(W_l Sigma_lr + W_r Sigma_rr),   Sigma_ii = D_i^-1 - Sigma_il W_l^T - Sigma_ir W_r^T
// Sigma_ii is written symmetrised.  Every adjacent pair of the level contains one odd node, so the pass writes the level's whole first
// off-diagonal into So (block (k, k+1) at k, column-major; So = NULL: not wanted).
__global__ void __launch_bounds__(128) k_bcr_selinv(int64_t m, int64_t stride, const double* Lc, const double* Za, const double* Zb, const double* Sc,
                                                    double* S, double* So) {
    __shared__ double sL[4][15 * 16], sT[4][5][225];   // [warp][W_l | W_r | Sigma_ll -> Sigma_il | Sigma_rr -> Sigma_ir | Sigma_lr -> Lc^-1 -> Sigma_ii]
    const int wib = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t t = (int64_t)blockIdx.x * 4 + wib;
    const int64_t i = 2 * t + 1;
    if (i >= m) return;
    const bool has_right = i + 1 < m;
    double *L = sL[wib], *Wl = sT[wib][0], *Wr = sT[wib][1], *Xl = sT[wib][2], *Xr = sT[wib][3], *Y = sT[wib][4];
    for (int k = lane; k < 225; k += 32) {
        const int r = k % 15, c = k / 15;
        if (r >= c) L[r * 16 + c] = Lc[t * 225 + k];
        Xl[k] = S[(i - 1) * stride * 225 + k];
        Xr[k] = has_right ? S[(i + 1) * stride * 225 + k] : 0.0;
        Y[k] = has_right ? Sc[t * 225 + k] : 0.0;
    }
    __syncwarp();
    if (lane < 30) {                                               // lanes 0..14: columns of W_l, 15..29: columns of W_r
        const int c = lane < 15 ? lane : lane - 15;
        double y[15];
#pragma unroll
        for (int r = 0; r < 15; r++) y[r] = lane < 15 ? Za[t * 225 + 15 * c + r] : (has_right ? Zb[t * 225 + 15 * c + r] : 0.0);
        bwd15(L, y);
        double* dst = (lane < 15 ? Wl : Wr) + 15 * c;
#pragma unroll
        for (int r = 0; r < 15; r++) dst[r] = y[r];
    }
    __syncwarp();
    double vl[8], vr[8];                                           // entry k = lane + 32 s of Sigma_il / Sigma_ir (column-major)
#pragma unroll
    for (int s = 0; s < 8; s++) {
        const int k = lane + 32 * s;
        if (k < 225) {
            const int a = k % 15, b = k / 15;
            double xl = 0.0, xr = 0.0;
#pragma unroll
            for (int q = 0; q < 15; q++) {
                xl = fma(-Wl[a + 15 * q], Xl[q + 15 * b], xl);
                xl = fma(-Wr[a + 15 * q], Y[b + 15 * q], xl);
                xr = fma(-Wl[a + 15 * q], Y[q + 15 * b], xr);
                xr = fma(-Wr[a + 15 * q], Xr[q + 15 * b], xr);
            }
            vl[s] = xl; vr[s] = xr;
        }
    }
    __syncwarp();
#pragma unroll
    for (int s = 0; s < 8; s++) {
        const int k = lane + 32 * s;
        if (k < 225) {
            const int a = k % 15, b = k / 15;
            Xl[k] = vl[s]; Xr[k] = vr[s];
            if (So) {
                So[(i - 1) * 225 + b + 15 * a] = vl[s];            // block (i-1, i) = Sigma_il^T
                if (has_right) So[i * 225 + k] = vr[s];            // block (i, i+1) = Sigma_ir
            }
        }
    }
    warp_inv_lower15(L, Y, lane);                                  // (its __syncwarp also publishes Sigma_il / Sigma_ir)
#pragma unroll
    for (int s = 0; s < 8; s++) {
        const int k = lane + 32 * s;
        if (k < 225) {
            const int a = k % 15, b = k / 15;
            double d = inv_entry15(Y, a, b);
#pragma unroll
            for (int q = 0; q < 15; q++) {
                d = fma(-Xl[a + 15 * q], Wl[b + 15 * q], d);
                d = fma(-Xr[a + 15 * q], Wr[b + 15 * q], d);
            }
            vl[s] = d;
        }
    }
    __syncwarp();
#pragma unroll
    for (int s = 0; s < 8; s++) { const int k = lane + 32 * s; if (k < 225) Y[k] = vl[s]; }
    __syncwarp();
    for (int k = lane; k < 225; k += 32) { const int a = k % 15, b = k / 15; S[i * stride * 225 + k] = 0.5 * (Y[k] + Y[b + 15 * a]); }
}

// ---- launchers ----------------------------------------------------------------------------------------------------------------------
cudaError_t whiten_launch(int rd, int64_t n, const double* records, const double* e, const double* H1, const double* H2, double* A1, double* A2, double* b, cudaStream_t st) {
    if (n == 0) return cudaSuccess;
    k_factor_whiten<<<(int)((n + 3) / 4), 128, 0, st>>>(n, rd, records, e, H1, H2, A1, A2, b);
    return cudaGetLastError();
}

cudaError_t chain_assemble_launch(int64_t nf, const double* G11, const double* G12, const double* G22, const double* g1, const double* g2, double lambda,
                                  int diagonal_damping, const double* prior_info, const double* prior_rhs, double* D, double* E, double* rhs, cudaStream_t st) {
    k_chain_assemble<<<(int)(nf + 1), 128, 0, st>>>(nf, G11, G12, G22, g1, g2, lambda, diagonal_damping, prior_info, prior_rhs, D, E, rhs);
    return cudaGetLastError();
}

// workspace layout: for every level l >= 1 the reduced system (D, E, b), for every level l >= 0 the eliminated nodes (Lc, Za, Zb, zb)
static int64_t bcr_doubles(int64_t m) {
    int64_t tot = 0;
    while (m > 1) {
        const int64_t odd = m / 2, even = (m + 1) / 2;
        tot += odd * (3 * 225 + 15);            // Lc, Za, Zb, zb of this level's odd nodes
        tot += even * (2 * 225 + 15);           // D, E, b of the next level
        m = even;
    }
    return tot + 16;
}
int64_t chain_solve_workspace_bytes(int64_t n_states) { return bcr_doubles(n_states) * 8; }

struct BcrLevel { int64_t m; double *Lc, *Za, *Zb, *zb, *En; };   // En: the reduced E' this level produces (the next level's E)

// forward sweep, two launches per level, down to one node; returns the number of levels and the root's D (and b)
static int bcr_forward(int64_t n_states, const double* D, const double* E, const double* b, double* ws, cudaStream_t st, BcrLevel* lv,
                       const double** root_D, const double** root_b) {
    int nl = 0;
    int64_t m = n_states;
    const double *cD = D, *cE = E, *cb = b;
    double* p = ws;
    while (m > 1) {
        const int64_t odd = m / 2, even = (m + 1) / 2;
        BcrLevel& L = lv[nl++];
        L.m = m;
        L.Lc = p; p += odd * 225; L.Za = p; p += odd * 225; L.Zb = p; p += odd * 225; L.zb = p; p += odd * 15;
        double* nD = p; p += even * 225; L.En = p; p += even * 225; double* nb = p; p += even * 15;
        k_bcr_eliminate<<<(int)((odd + 3) / 4), 128, 0, st>>>(m, cD, cE, cb, L.Lc, L.Za, L.Zb, L.zb);
        k_bcr_reduce<<<(int)((even + 3) / 4), 128, 0, st>>>(m, cD, cb, L.Za, L.Zb, L.zb, nD, L.En, nb);
        cD = nD; cE = L.En; cb = b ? nb : nullptr; m = even;
    }
    *root_D = cD; *root_b = cb;
    return nl;
}

cudaError_t chain_solve_launch(int64_t n_states, const double* D, const double* E, const double* b, double* x, double* ws, cudaStream_t st, int* launches) {
    BcrLevel lv[64];
    const double *rD, *rb;
    const int nl = bcr_forward(n_states, D, E, b, ws, st, lv, &rD, &rb);
    k_bcr_root<<<1, 32, 0, st>>>(rD, rb, x, 1);
    int64_t stride = (int64_t)1 << nl;
    for (int l = nl - 1; l >= 0; l--) {
        stride >>= 1;
        const int64_t odd = lv[l].m / 2;
        k_bcr_backsub<<<(int)((odd + 3) / 4), 128, 0, st>>>(lv[l].m, stride, lv[l].Lc, lv[l].Za, lv[l].Zb, lv[l].zb, x);
    }
    if (launches) *launches = 3 * nl + 1;
    return cudaGetLastError();
}

// Same workspace as the solve.  A level's reduced E' is dead once the forward sweep is done; its slot then holds that level's Sigma
// off-diagonal blocks (written by the level's selected-inversion pass, read by the next finer one).  Level 0's go to S_off.
cudaError_t chain_marginals_launch(int64_t n_states, const double* D, const double* E, double* S_diag, double* S_off, double* ws, cudaStream_t st,
                                   int* launches) {
    BcrLevel lv[64];
    const double *rD, *rb;
    const int nl = bcr_forward(n_states, D, E, nullptr, ws, st, lv, &rD, &rb);
    k_bcr_root_inv<<<1, 32, 0, st>>>(rD, S_diag);
    int64_t stride = (int64_t)1 << nl;
    for (int l = nl - 1; l >= 0; l--) {
        stride >>= 1;
        const int64_t odd = lv[l].m / 2;
        k_bcr_selinv<<<(int)((odd + 3) / 4), 128, 0, st>>>(lv[l].m, stride, lv[l].Lc, lv[l].Za, lv[l].Zb, lv[l].En, S_diag, l > 0 ? lv[l - 1].En : S_off);
    }
    if (launches) *launches = 3 * nl + 1;
    return cudaGetLastError();
}

}  // namespace cpi
