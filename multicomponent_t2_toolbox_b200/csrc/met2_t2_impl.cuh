// met2_t2_impl.cuh — the T2 fit kernel template and its launch helpers (included by met2_t2.cu and by one translation
// unit per regularisation method, so that every method gets its own lean kernel: the instruction footprint of the hot
// loop has to stay inside the 128 KB instruction cache — profiles/r01_t2_fit_v4_ncu_summary.txt shows what happens
// otherwise: "no_instruction" becomes the top stall).
#pragma once
#include <cmath>
#include <cstdlib>

#include "met2_device.cuh"
#include "met2_host.h"

namespace met2 {

constexpr int T2_TILE_MAX = 512;    // largest tile (voxels of one FA index handed to a CTA at once)
constexpr int T2_TILE_MIN = 32;     // tail tiles

struct T2Args {
    const double* sig;
    const int* fa_index;
    long long V;
    met2_t2_cfg cfg;
    const double *dic, *dicT, *G, *kband, *lambdas, *logT2;
    const unsigned char* comp;
    const double *red_basis, *red_coef;   // reduced echo basis U [nA][nTE][RD] and coefficients C [nA][nT2][RD]
                                          // (met2_echo_basis); only the echo-space kernels read them
    double *fsol, *est, *reg, *maps;
    unsigned* status;
    // workspace
    int* hist;        // [nA]
    int* cursor;      // [nA]
    int* bin_start;   // [nA + 1]
    int* perm;        // [V]
    int* tile_fa;     // [max tiles]
    int* tile_start;
    int* tile_cnt;
    int* counters;    // [0] = number of tiles, [1] = next tile
    int pmax;
    int warps;
    // shared full-set factor tables (X2 with MET2_T2_FLAG_FULL_START): the first T2_NTAB abscissae of bounded Brent do
    // not depend on the voxel, so the inverse Cholesky factor of the FULL column set, (G_a + lam_j K)^-1 = T T^T, is
    // built once per (flip angle, abscissa) by t2_full_factors_kernel and copied instead of being re-derived per voxel
    const double* tfull;     // [ntab][nA][tri(nT2)], first entry NaN if not positive definite.  X2: inverse Cholesky
                             // factors T; BayesReg: the Cholesky factors U themselves (evidence)
    const double* lam_tab;   // [ntab]
    int ntab;                // tables built
    int ntab_use;            // how many of them the NNLS full-set starts consult
    double lcurve_switch;    // echo-space L-curve: grid points below this lambda are solved in the Gram domain
                             // (met2_t2_echo_reg_impl.cuh); MET2_LCURVE_SWITCH overrides it (met2_host.h)
};

constexpr int T2_NTAB_X2 = 3;      // measured on config 2 (T2 stage): no table 444 ms, 2 tables 398, 3 tables 390, 4 tables 390
constexpr int T2_NTAB_BAYES = 9;   // BayesReg: the evidence needs the FULL-set factor at every abscissa, so every tabulated
                                   // abscissa saves a whole n x n factorisation (bayes_cost)
constexpr int T2_NTAB_MAX = 16;
constexpr double T2_LCURVE_SWITCH = 1e-5;   // see T2Args::lcurve_switch

// ---------------------------------------------------------------------------------------------- L-curve corner
// Triangle method of algorithms.py:150-206 (select_corner + scale_curve) on curves of length nl at S[oLx..], S[oLy..].
__device__ __forceinline__ int select_corner_warp(int oLx, int oLy, int nl, int lane) {
    // scale both curves to [-10, 10]: ((u-l)/(vmax-vmin)) * (a - (u*vmin - l*vmax)/(u-l))
    for (int c = 0; c < 2; ++c) {
        const int oA = c ? oLy : oLx;
        double vmin = INFINITY, vmax = -INFINITY;
        bool has_nan = false;
        for (int i = lane; i < nl; i += 32) {
            double v = S[oA + i];
            if (v != v) has_nan = true;
            vmin = fmin(vmin, v);
            vmax = fmax(vmax, v);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            vmin = fmin(vmin, __shfl_xor_sync(FULL_MASK, vmin, o));
            vmax = fmax(vmax, __shfl_xor_sync(FULL_MASK, vmax, o));
        }
        if (__any_sync(FULL_MASK, has_nan)) vmin = vmax = NAN;   // numpy min/max propagate NaN
        double scale = 20.0 / (vmax - vmin);
        double shift = (10.0 * vmin - (-10.0) * vmax) / 20.0;
        __syncwarp();
        for (int i = lane; i < nl; i += 32) S[oA + i] = scale * (S[oA + i] - shift);
        __syncwarp();
    }
    const double cte = 7.0 * 3.141592653589793 / 8.0;
    const double cx = S[oLx + nl - 1], cy = S[oLy + nl - 1];
    double best_ang = INFINITY;
    int best_ord = -1;
    for (int k = lane; k < nl - 2; k += 32) {
        double bx = S[oLx + k], by = S[oLy + k];
        for (int j = k + 1; j < nl - 1; ++j) {
            double ax = S[oLx + j], ay = S[oLy + j];
            double dx1 = ax - bx, dy1 = ay - by;
            double ab = sqrt(dx1 * dx1 + dy1 * dy1);
            double dx2 = ax - cx, dy2 = ay - cy;
            double ac = sqrt(dx2 * dx2 + dy2 * dy2);
            double dx3 = bx - cx, dy3 = by - cy;
            double bc = sqrt(dx3 * dx3 + dy3 * dy3);
            double cosa = (ab * ab + ac * ac - bc * bc) / (2.0 * ab * ac);
            // Python: max(-1.0, min(cosa, 1.0)) -> NaN becomes -1.0
            if (cosa != cosa) cosa = -1.0;
            else cosa = fmax(-1.0, fmin(cosa, 1.0));
            double ang = acos(cosa);
            double area = 0.5 * ((bx - ax) * (ay - cy) - (ax - cx) * (by - ay));
            if (area > 0.0 && ang < cte && ang < best_ang) {
                best_ang = ang;
                best_ord = k * nl + j;
            }
        }
    }
    // global minimum angle; ties -> earliest (k, j) in the reference's loop order
    unsigned long long key = (best_ord >= 0) ? (unsigned long long)__double_as_longlong(best_ang + 0.0) : ~0ull;
    unsigned hi = (unsigned)(key >> 32), lo = (unsigned)key;
    unsigned mhi = __reduce_min_sync(FULL_MASK, hi);
    unsigned mlo = __reduce_min_sync(FULL_MASK, (hi == mhi) ? lo : 0xffffffffu);
    if (mhi == 0xffffffffu && mlo == 0xffffffffu) return nl - 1;
    bool win = (best_ord >= 0) && hi == mhi && lo == mlo;
    unsigned ord = __reduce_min_sync(FULL_MASK, win ? (unsigned)best_ord : 0xffffffffu);
    return (int)(ord % (unsigned)nl);
}

// ---------------------------------------------------------------------------------------------- BayesReg objective
// -log evidence of bayesian_interpolation.py:107-126 for one lambda (= x), given the Tikhonov-NNLS solution f in
// column space (S[W.xc..]):  A = beta*B + (beta*x)*K, U = chol(A) (upper), and
//   cost = beta*ED + beta*x*EW + log(prod diag U) - (n/2) log(pi/2) - sum log(1 + erf(U f / sqrt 2))
//        + (m/2) log(2 pi) - (m/2) log(beta) + (n/2) log(pi) - (n/2) log(2 beta x) - log(det L).
// U itself (n x n, natural column order) is built in the warp's T region (free between NNLS solves) by the blocked
// FP64-tensor-core Cholesky chol_upper_blocked; log det U = log prod U_kk and U f is one triangular mat-vec — the same
// quantities, formed the same way, as the reference's.  (Round 1 used the inverse factor: U f = T^T (A f).  Together
// with the ~1e-9 relative error of the Gram-domain NNLS solution that put 25 % of the config-4 voxels more than 1e-6
// away from the reference's lambda, where the reference's own reproducibility under a 1e-13 perturbation is 5 %.)
template <int NS, bool GSH>
__device__ __forceinline__ double bayes_cost(const Slots<NS>& W, int oG, const double* __restrict__ Gg, int ldg, int oKb,
                                             int n, int m, int lane, double x, double beta, double sse, double nrm,
                                             double log_det_L, unsigned& st, const double* __restrict__ utab) {
    const int oT = W.T;
    const double bx = beta * x;
    // While Brent is still on its voxel-independent golden chain (the first T2_NTAB_BAYES abscissae, bracket wider than
    // ~1e-2), the factor U0 of B + x K comes from the shared tables (utab) and U = sqrt(beta) U0; afterwards A is
    // factored here, with beta inside the matrix like the reference's cholesky(beta*B + beta*x*K).  The two differ by
    // rounding only, which is why the tables stop before the convergence phase: there Brent compares nearly equal
    // evidences and a 1e-16 change of the objective can move lambda by 1e-3 relative (measured with 16 tables: 2 of
    // 2 048 voxels; with 9: none).
    bool pd = true;
    if (utab) {
        const double sb = sqrt(beta);
        for (int i = lane; i < tri(n); i += 32) S[oT + i] = __ldg(utab + i) * sb;
        __syncwarp();
    } else {
        auto Aent = [&](int r, int c) -> double {
            double a = beta * (GSH ? S[oG + r * ldg + c] : __ldg(Gg + r * ldg + c));
            const int d = r - c + 2;   // K[r][c] = kband[d][c]
            if (d >= 0 && d <= 4) a = a + bx * S[oKb + d * n + c];
            return a;
        };
        pd = chol_upper_blocked<NS>(W, Aent, n, lane);
    }
    if (!pd) st |= MET2_ST_NOT_PD;
    // det_U = prod(diag(U))  (np.prod order)
    double det_u = 1.0;
    for (int k = 0; k < n; ++k) det_u *= S[oT + tri(k) + k];
    // U f: row k of U times f (natural order; f = S[W.xc ..], zeros outside the support)
    double uf[NS];
    tmul<NS>(oT, W.xc, n, lane, uf);
    double series = 0.0;
#pragma unroll
    for (int t = 0; t < NS; ++t) {
        const int i = lane + 32 * t;
        if (i < n) series += log(1.0 + erf(0.7071067811865475 * uf[t]));
    }
    series = warp_sum(series);
    const double ED = 0.5 * sse, EW = 0.5 * nrm;
    const double PI = 3.141592653589793;
    const double hn = n / 2.0, hm = m / 2.0;
    const double cost1 = beta * ED + beta * x * EW + log(det_u) - hn * log(PI / 2.0) - series;
    const double cost2 = hm * log(2.0 * PI) - hm * log(beta) + hn * log(PI) - hn * log(2.0 * beta * x) - log_det_L;
    return pd ? (cost1 + cost2) : INFINITY;
}

// ---------------------------------------------------------------------------------------------- GCV objective
// obj_nnls_gcv of algorithms.py:285-296, quirks included: with sel = {f > 0} (k columns), Dr = D[:, sel] and the SCALAR
// s = sum_sel L_ii^2 (the reference's L[f>0, f>0] picks diagonal entries), the reference forms Mk = Dr^T Dr + x s 1 1^T
// (x s added to EVERY entry), A = Dr lstsq(Mk, Dr^T, rcond=None) and returns log( (SSEr^2/m) / ((m - tr A)/m)^2 ) with
// SSEr the residual norm of the STACKED system.  lstsq (gelsd) is a truncated pseudo-inverse: singular values <= eps*k*s_max
// are dropped.  With the symmetric eigen-decomposition Mk = U diag(mu) U^T:  tr A = sum_kept (1 - x s (1^T u_i)^2 / mu_i).
//
// Mk is numerically of rank 10-17 whatever k is (the EPG dictionary's singular values fall by ~12x per index), so the
// k x k eigenproblem is first reduced by a rank-revealing (diagonally pivoted) Cholesky factorisation Mk = C C^T + E,
// C: k x r, stopped when the largest residual diagonal entry is below 1e-16 of the largest diagonal entry (far under the
// eps*k*mu_max cut-off).  The non-zero spectrum of C C^T is that of the r x r matrix H = C^T C = W diag(mu) W^T, with
// u_i = C w_i / sqrt(mu_i), hence  tr A = sum_kept (1 - x s (g^T w_i)^2 / mu_i^2),  g = C^T 1.
// H goes through a parallel (round-robin) two-sided Jacobi iteration that carries g along as one row of W.
// tools/proto_gcv_pivchol.py (CPU) measured the reduced form against the full k x k eigen-decomposition: identical
// objective statistics against the reference (median |d obj| 5e-7 .. 8e-6; r <= 17 on the phantom).
// SURVEY.md a-8: the kept/dropped decision sits at rounding level for eigenvalues near eps*k*mu_max, so the reference
// itself is not reproducible there; parity for GCV is statistical (DESIGN.md "Parity").
constexpr int GCV_RCAP = 20;              // columns of C (numerical rank cap)
constexpr int GCV_LDC = GCV_RCAP + 1;     // odd row stride: conflict-free column walks
__host__ __device__ __forceinline__ int gcv_region_doubles(int n) { return n * GCV_LDC + GCV_RCAP * (GCV_RCAP | 1); }

template <int NS>
__device__ __forceinline__ double jacobi_trace(const Slots<NS>& W, int oA, int N, double xs_scale, int k_sel, int lane,
                                               int& kept) {
    // matrix H: N x N row-major with stride LD at S[oA ..]; functional e at S[W.rs ..]; (c, s) of a round at S[W.gs ..]
    const int LD = N | 1;
    const int Ne = N + (N & 1);
    const int half = Ne >> 1;
    // an off-diagonal entry below 1e-18 of the largest diagonal entry moves no eigenvalue by more than that, four
    // orders of magnitude under the eps*k*l_max cut-off; without the floor the noise-level block keeps rotating
    double dmax = 0.0;
    for (int i = lane; i < N; i += 32) dmax = fmax(dmax, fabs(S[oA + i * LD + i]));
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) dmax = fmax(dmax, __shfl_xor_sync(FULL_MASK, dmax, o));
    const double floor_abs = 1e-18 * dmax;
    for (int sweep = 0; sweep < 14; ++sweep) {
        double off = 0.0;
        for (int round = 0; round < Ne - 1; ++round) {
            // ---- rotation of pair `lane` of this round (circle method)
            int pp = -1, qq = -1;
            if (lane < half) {
                if (lane == 0) {
                    pp = round;
                    qq = Ne - 1;
                } else {
                    pp = round + lane;
                    if (pp >= Ne - 1) pp -= Ne - 1;
                    qq = round - lane + (Ne - 1);
                    if (qq >= Ne - 1) qq -= Ne - 1;
                }
                if (pp > qq) {
                    int tmp = pp;
                    pp = qq;
                    qq = tmp;
                }
                if (qq >= N) pp = qq = -1;
            }
            double c = 1.0, s = 0.0;
            if (pp >= 0) {
                const double apq = S[oA + pp * LD + qq];
                const double app = S[oA + pp * LD + pp], aqq = S[oA + qq * LD + qq];
                if (fabs(apq) > 1.1e-16 * sqrt(fabs(app * aqq)) && fabs(apq) > floor_abs) {   // relative criterion
                    off += apq * apq;
                    const double zeta = (aqq - app) / (2.0 * apq);
                    const double tt = ((zeta >= 0.0) ? 1.0 : -1.0) / (fabs(zeta) + sqrt(1.0 + zeta * zeta));
                    c = 1.0 / sqrt(1.0 + tt * tt);
                    s = tt * c;
                }
                // the functional transforms like a row of W: e_p' = c e_p - s e_q, e_q' = s e_p + c e_q  (identity, and
                // no write at all, for a skipped rotation: a round without rotations touches no shared memory)
                if (s != 0.0) {
                    const double ep = S[W.rs + pp], eq = S[W.rs + qq];
                    S[W.rs + pp] = c * ep - s * eq;
                    S[W.rs + qq] = s * ep + c * eq;
                }
            }
            // a round in which no pair rotates changes nothing (the last sweep consists of such rounds only)
            if (!__any_sync(FULL_MASK, s != 0.0)) continue;
            if (lane < half) {
                S[W.gs + 3 * lane] = c;
                S[W.gs + 3 * lane + 1] = s;
                SI(W.gs + 3 * lane + 2, 0) = pp;
                SI(W.gs + 3 * lane + 2, 1) = qq;
            }
            __syncwarp();
            // ---- columns: H <- H J.  Two rotations per pass: half-warp `sub` takes pair i0 + sub, its 16 lanes the rows
            //      (N <= 20, so at most two rows per lane); the pairs of a round touch disjoint columns
            const int sub = lane >> 4, l16 = lane & 15;
            for (int i0 = 0; i0 < half; i0 += 2) {
                const int i = i0 + sub;
                if (i < half) {
                    const int p2 = SI(W.gs + 3 * i + 2, 0), q2 = SI(W.gs + 3 * i + 2, 1);
                    const double ci = S[W.gs + 3 * i], si = S[W.gs + 3 * i + 1];
                    if (p2 >= 0 && si != 0.0) {   // a skipped rotation is exactly the identity (c = 1, s = 0): nothing to do
                        for (int r = l16; r < N; r += 16) {
                            const double xv = S[oA + r * LD + p2], yv = S[oA + r * LD + q2];
                            S[oA + r * LD + p2] = ci * xv - si * yv;
                            S[oA + r * LD + q2] = si * xv + ci * yv;
                        }
                    }
                }
            }
            __syncwarp();
            // ---- rows: H <- J^T H   (16 lanes = columns)
            for (int i0 = 0; i0 < half; i0 += 2) {
                const int i = i0 + sub;
                if (i < half) {
                    const int p2 = SI(W.gs + 3 * i + 2, 0), q2 = SI(W.gs + 3 * i + 2, 1);
                    const double ci = S[W.gs + 3 * i], si = S[W.gs + 3 * i + 1];
                    if (p2 >= 0 && si != 0.0) {
                        for (int cc = l16; cc < N; cc += 16) {
                            const double xv = S[oA + p2 * LD + cc], yv = S[oA + q2 * LD + cc];
                            S[oA + p2 * LD + cc] = ci * xv - si * yv;
                            S[oA + q2 * LD + cc] = si * xv + ci * yv;
                        }
                    }
                }
            }
            __syncwarp();
        }
        off = warp_sum(off);
        if (off == 0.0) break;
    }
    // eigenvalues on the diagonal; truncated-pseudo-inverse trace
    double lmax = 0.0;
    for (int i = lane; i < N; i += 32) lmax = fmax(lmax, S[oA + i * LD + i]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) lmax = fmax(lmax, __shfl_xor_sync(FULL_MASK, lmax, o));
    const double tau = 2.220446049250313e-16 * (double)k_sel * lmax;
    double tr = 0.0;
    int nk = 0;
    for (int i = lane; i < N; i += 32) {
        const double li = S[oA + i * LD + i];
        if (li > tau) {
            const double ei = S[W.rs + i];
            tr += 1.0 - xs_scale * (ei * ei) / (li * li);
            ++nk;
        }
    }
    kept = __reduce_add_sync(FULL_MASK, nk);     // eigenvalues above the cut-off = rank of the truncated pseudo-inverse
    return warp_sum(tr);
}

template <int NS, bool GSH>
__device__ __forceinline__ double gcv_cost(const Slots<NS>& W, int oG, const double* __restrict__ Gg, int ldg, int oLb,
                                           int n, int m, int lane,
                                           double x, double sse, double nrm, int p, int& kept) {
    // ---- sel = positions with a strictly positive coefficient (after an itmax stop some may be 0), compacted as
    //      column indices into S[W.gs ..] (ints); row i of Mk <-> lane i % 32, slot i / 32
    __syncwarp();
    int k = 0;
    double sdiag = 0.0;
#pragma unroll
    for (int t = 0; t < NS; ++t) {
        const int i = lane + 32 * t;
        const bool in = (i < p) && (S[W.xs + i] > 0.0);
        const unsigned bal = __ballot_sync(FULL_MASK, in);
        if (in) {
            const int cidx = SI(W.ix, i);
            SI(W.gs, k + __popc(bal & ((1u << lane) - 1u))) = cidx;
            const double lii = S[oLb + 2 * n + cidx];
            sdiag = fma(lii, lii, sdiag);
        }
        k += __popc(bal);
    }
    sdiag = warp_sum(sdiag);
    __syncwarp();
    const double xs = x * sdiag;
    const int oC = W.T, oH = W.T + k * GCV_LDC;
    // ---- diagonally pivoted Cholesky  Mk ~ C C^T  (residual diagonal in S[W.rs ..])
    int col[NS];
    unsigned done = 0u;
    double dmax = 0.0;
#pragma unroll
    for (int t = 0; t < NS; ++t) {
        const int i = lane + 32 * t;
        col[t] = (i < k) ? SI(W.gs, i) : 0;
        if (i < k) {
            const double d = (GSH ? S[oG + col[t] * ldg + col[t]] : __ldg(Gg + col[t] * ldg + col[t])) + xs;
            S[W.rs + i] = d;
            dmax = fmax(dmax, d);
        } else {
            done |= 1u << t;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) dmax = fmax(dmax, __shfl_xor_sync(FULL_MASK, dmax, o));
    const double thr = 1e-16 * dmax;
    __syncwarp();
    int r = 0;
    for (; r < GCV_RCAP && r < k; ++r) {
        double bv = 0.0;
        int bj = -1;
#pragma unroll
        for (int t = 0; t < NS; ++t) {
            const int i = lane + 32 * t;
            if (!((done >> t) & 1u)) {
                const double d = S[W.rs + i];
                if (d > bv) {
                    bv = d;
                    bj = i;
                }
            }
        }
        const int piv = warp_argmax_pos(bv, bj);
        if (piv < 0) break;
        const double dp = S[W.rs + piv];
        if (!(dp > thr)) break;
        const int cp = SI(W.gs, piv);
        const double rinv = rsqrt_fast(dp);
#pragma unroll
        for (int t = 0; t < NS; ++t) {
            const int i = lane + 32 * t;
            if (i < k) {
                double cv = 0.0;
                if (i == piv) {
                    cv = dp * rinv;
                    done |= 1u << t;
                } else if (!((done >> t) & 1u)) {
                    double v = (GSH ? S[oG + cp * ldg + col[t]] : __ldg(Gg + cp * ldg + col[t])) + xs;
                    for (int l = 0; l < r; ++l) v = fma(-S[oC + i * GCV_LDC + l], S[oC + piv * GCV_LDC + l], v);
                    cv = v * rinv;
                    S[W.rs + i] = fma(-cv, cv, S[W.rs + i]);
                }
                S[oC + i * GCV_LDC + r] = cv;
            }
        }
        __syncwarp();
    }
    // ---- H = C^T C (r x r) and g = C^T 1
    // every lane has read the residual diagonal (S[W.rs + piv] above) before g overwrites S[W.rs ..]: without this
    // barrier the loop exit was a write-after-read race between lanes (found by the SIMT emulator's sequential lane
    // schedule, tests/emu; harmless while the warp runs in lockstep, which is what the GPU did)
    __syncwarp();
    const int LD = r | 1;
    for (int a = 0; a < r; ++a) {
        const int b = a + lane;
        if (b < r) {
            double h = 0.0;
            for (int i = 0; i < k; ++i) h = fma(S[oC + i * GCV_LDC + a], S[oC + i * GCV_LDC + b], h);
            S[oH + a * LD + b] = h;
            S[oH + b * LD + a] = h;
        }
    }
    if (lane < r) {
        double g = 0.0;
        for (int i = 0; i < k; ++i) g += S[oC + i * GCV_LDC + lane];
        S[W.rs + lane] = g;
    }
    __syncwarp();
    kept = 0;
    const double tr = (r > 0) ? jacobi_trace<NS>(W, oH, r, xs, k, lane, kept) : 0.0;
    const double dm = (double)m;
    const double num = (1.0 / dm) * (sse + x * nrm);
    const double den = (1.0 / dm) * (dm - tr);
    return log(num / (den * den));
}

// ---------------------------------------------------------------------------------------------- full-set factor tables
// One warp per (abscissa j, flip angle a).  The abscissae are produced by the same Brent state machine the fit kernel
// runs (so the fit kernel can match them bit for bit), fed with the objective f(x) = x: x0 = a + g (b - a), x1 = the
// golden step to the right of it (worse), then golden steps to the left, each better than the last — the path of every
// voxel whose optimum is small compared with the bracket, for as long as its parabolic steps are rejected.  A voxel
// that leaves this path simply stops matching the table.
template <int NS>
__global__ void __launch_bounds__(32) t2_full_factors_kernel(const double* __restrict__ G, const double* __restrict__ kband,
                                                             int n, int nA, double lo, double hi, double xatol,
                                                             int maxfun, int upper, double* __restrict__ tfull,
                                                             double* __restrict__ lam_tab) {
    const int lane = threadIdx.x;
    const int a = blockIdx.x % nA, j = blockIdx.x / nA;
    Brent B;
    double lam = B.start(lo, hi, xatol, maxfun);
    bool more = true;
    for (int q = 0; q < j; ++q) {
        const double f = lam;
        if (more) more = B.feed(f, lam);
    }
    const double lj = more ? lam : NAN;
    if (a == 0 && lane == 0) lam_tab[j] = lj;
    Slots<NS> W;
    W.carve(0, n);
    const double* Ga = G + (size_t)a * n * n;
    auto Aent = [&](int r, int c) -> double {
        double v = __ldg(Ga + r * n + c);
        const int d = r - c + 2;   // K[r][c] = kband[d][c]
        if (d >= 0 && d <= 4) v = fma(lj, __ldg(kband + d * n + c), v);
        return v;
    };
    // upper: the Cholesky factor U itself (BayesReg evidence); otherwise the inverse factor T (X2 full-set starts)
    const bool pd = (lj == lj) && (upper ? chol_upper_blocked<NS>(W, Aent, n, lane) : rebuild_T_blocked<NS>(W, Aent, n, lane));
    double* out = tfull + ((size_t)j * nA + a) * tri(n);
    for (int i = lane; i < tri(n); i += 32) out[i] = S[W.T + i];
    __syncwarp();
    if (!pd && lane == 0) out[0] = NAN;
}

// ---------------------------------------------------------------------------------------------- fit kernel
// shared-memory layout in doubles: [G n*n][K band 5n][L band 5n][logT2 n][lambdas 64][comp n bytes -> (n+7)/8]
// then per warp: [NNLS slots][signal 64][L-curve curves 2 x 64 | Brent-best snapshot 48 NS]
__host__ __device__ __forceinline__ int t2_ldg(int n) { return (n + 1) & ~1; }   // even row stride: 16-byte aligned rows
// The Gram matrix of the tile's flip angle is staged in shared memory for nT2 <= 64 only.  For the wide grids (96 bins:
// 74 KB, 100 bins: 80 KB) it stays in global memory (read-only path, L1/L2-resident: every warp of the CTA works on the
// same flip angle): the per-voxel factor is 37-40 KB there and the staged copy cost half of the resident warps — config 4
// (BayesReg-InvT2, 100 bins) ran at TWO warps per SM (profiles/r02_config4_ncu_summary.txt).
__host__ __device__ constexpr __forceinline__ bool t2_gram_in_shared(int ns) { return ns <= 2; }
__host__ __device__ __forceinline__ int t2_table_doubles(int n, bool gsh) {
    return ((gsh ? n * t2_ldg(n) : 0) + 10 * n + n + MET2_MAX_LAMBDAS + (n + 7) / 8 + 31) & ~31;
}

template <int NS>
__host__ __device__ __forceinline__ int t2_warp_doubles(int pmax) {
    // + signal (64) + the L-curve curves (2 x 64), which double as the Brent-best snapshot (x: 32 NS, ix: 16 NS)
    return (Slots<NS>::doubles(pmax) + 64 + (48 * NS > 128 ? 48 * NS : 128) + 31) & ~31;
}

constexpr int T2_MAX_THREADS = 320;

// METHOD (MET2_REG_*) is a template parameter: each regularisation method compiles to its own kernel.
template <int NS, int ME, int METHOD>
__global__ void __launch_bounds__(T2_MAX_THREADS, 1) t2_fit_kernel(T2Args A) {
    __shared__ int s_tile, s_next;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int n = A.cfg.nT2, m = A.cfg.nTE;
    constexpr int method = METHOD;
    // position slots of the solver: a plain solve has at most min(nT2, nTE) <= 32 ME positive columns
    constexpr int PS = (METHOD == MET2_REG_NNLS && ME < NS) ? ME : NS;
    constexpr bool GSH = t2_gram_in_shared(NS);
    const int oG = 0;
    const int ldg = GSH ? t2_ldg(n) : n;         // row stride of G where the solver reads it
    const int oKb = GSH ? oG + n * ldg : 0;      // K band rows 0..4
    const int oLb = oKb + 5 * n;         // L band rows 0..4
    const int oLogT2 = oLb + 5 * n;
    const int oLam = oLogT2 + n;
    unsigned char* scomp = reinterpret_cast<unsigned char*>(S + oLam + MET2_MAX_LAMBDAS);
    const int wbase = t2_table_doubles(n, GSH) + warp * t2_warp_doubles<NS>(A.pmax);
    Slots<NS> W;
    W.carve(wbase, A.pmax);
    const int oM = wbase + Slots<NS>::doubles(A.pmax);
    const int oLx = oM + 64, oLy = oLx + 64;

    for (int i = threadIdx.x; i < 10 * n; i += blockDim.x) S[oKb + i] = A.kband ? A.kband[i] : 0.0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        S[oLogT2 + i] = A.logT2[i];
        scomp[i] = A.comp[i];
    }
    for (int i = threadIdx.x; i < MET2_MAX_LAMBDAS; i += blockDim.x)
        S[oLam + i] = (A.lambdas && i < A.cfg.nLambda) ? A.lambdas[i] : 0.0;
    const int ntiles = A.counters[0];

    while (true) {
        __syncthreads();   // previous tile fully consumed (G, s_next) before they are overwritten
        if (threadIdx.x == 0) {
            s_tile = atomicAdd(&A.counters[1], 1);
            s_next = 0;
        }
        __syncthreads();
        const int tile = s_tile;
        if (tile >= ntiles) break;
        const int fa = A.tile_fa[tile];
        const int tstart = A.tile_start[tile], tcnt = A.tile_cnt[tile];
        const double* Gg = A.G + (size_t)fa * n * n;
        if (GSH) {
            for (int i = threadIdx.x; i < n * n; i += blockDim.x) {
                const int r = i / n;
                S[oG + r * ldg + (i - r * n)] = __ldg(Gg + i);
            }
        }
        __syncthreads();
        const double* D = A.dic + (size_t)fa * m * n;
        const double* Dt = A.dicT + (size_t)fa * n * m;

        while (true) {
            int it = 0;
            if (lane == 0) it = atomicAdd(&s_next, 1);
            it = __shfl_sync(FULL_MASK, it, 0);
            if (it >= tcnt) break;
            const long long v = A.perm[tstart + it];
            // ---- load, validity (motor...:124-131), normalise by km = M[0]
            unsigned st = load_signal<ME>(A.sig, v, m, oM, lane);
            const int fav = A.fa_index[v];
            const bool normalise = !(A.cfg.flags & MET2_T2_FLAG_NO_NORMALISE);
            const double km = normalise ? S[oM] : 1.0;
            if (!st && (!(km > 0.0) || fav < 0 || fav >= A.cfg.nA)) st = MET2_ST_SKIPPED;
            double regv = 0.0;
            int p = 0;
            double fit[ME];
#pragma unroll
            for (int u = 0; u < ME; ++u) fit[u] = 0.0;
            if (!st) {
                __syncwarp();
#pragma unroll
                for (int u = 0; u < ME; ++u) {
                    int e = lane + 32 * u;
                    if (e < m) S[oM + e] = S[oM + e] / km;
                }
                __syncwarp();
                compute_c<NS>(W, D, oM, m, n, lane);
                set_dspace<NS>(W, Dt, oM, lane);
                // ---- lambda-search driver: a small state machine around ONE inlined NNLS call site.
                //   NNLS     : plain solve                                                    (algorithms.py:55)
                //   T2SPARC  : one Tikhonov solve at lambda_fixed                             (algorithms.py:262)
                //   X2       : plain solve -> SSE; Brent on |SSE(lam) - factor*SSE|/SSE; final (algorithms.py:211-233)
                //   L_curve  : grid of nLambda solves -> curves -> corner; final               (algorithms.py:88-113)
                enum { ST_PLAIN0 = 0, ST_SEARCH = 1, ST_FINAL = 2 };
                int stage;
                bool reg;
                double lam = 0.0, SSE = 0.0;
                int gi = 0;
                Brent B;
                if (method == MET2_REG_NNLS) {
                    stage = ST_FINAL; reg = false;
                } else if (method == MET2_REG_T2SPARC) {
                    stage = ST_FINAL; reg = true; lam = A.cfg.lambda_fixed;
                } else if (method == MET2_REG_X2 || method == MET2_REG_BAYESREG) {
                    stage = ST_PLAIN0; reg = false;
                } else if (method == MET2_REG_GCV) {
                    stage = ST_SEARCH; reg = true;
                    lam = B.start(A.cfg.brent_lo, A.cfg.brent_hi, A.cfg.brent_xatol, A.cfg.maxfun);
                    if (A.cfg.flags & MET2_T2_FLAG_GCV_EVAL) {   // objective-level parity hook: one solve at lambda_fixed
                        stage = ST_FINAL;
                        lam = A.cfg.lambda_fixed;
                    } else if (A.cfg.flags & MET2_T2_FLAG_GCV_GRID) {   // arg-min of the objective over the lambda grid
                        lam = S[oLam];
                    }
                } else {   // MET2_REG_LCURVE
                    stage = ST_SEARCH; reg = true; lam = S[oLam];
                }
                int nst = 0;
                double beta = 0.0;
                const bool warm = !(A.cfg.flags & MET2_T2_FLAG_COLD_START);
                p = 0;
                // X2 with L = I: Brent's first abscissa (3.82 on [0, 10]) gives a solution with nearly every column
                // active, so that solve starts from the FULL set with the feasible point x_j = c_j / (G + lam K)_jj and
                // lets the secondary loop drop the few columns that do not belong, instead of ~55 single-column appends.
                // (Host sets MET2_T2_FLAG_FULL_START only for the identity matrix: with InvT2 the long-T2 columns are
                // barely penalised and most of them leave again — measured 2x slower for T2SPARC.)
                bool t_ready = false;
                auto full_set_start = [&](double lam0) {
#pragma unroll
                    for (int tt = 0; tt < NS; ++tt) {
                        const int j = lane + 32 * tt;
                        if (j < n) {
                            const double djj = fma(lam0, S[oKb + 2 * n + j], GSH ? S[oG + j * ldg + j] : __ldg(Gg + j * ldg + j));
                            SI(W.ix, j) = j;
                            S[W.xs + j] = fmax(S[W.cc + j] / djj, 1e-300);
                        }
                    }
                    __syncwarp();
                    p = n;
                };
                // If lam is one of the tabulated (voxel-independent) Brent abscissae, start its solve from the full set
                // with the shared factor of this flip angle instead of re-deriving a factor for the carried-over set.
                auto try_table = [&](double lam0) {
                    t_ready = false;
                    if (!A.tfull || !warm) return;
                    int jt = -1;
#pragma unroll
                    for (int q = 0; q < A.ntab_use; ++q)
                        if (lam0 == __ldg(A.lam_tab + q)) jt = q;
                    if (jt < 0) return;
                    const double* src = A.tfull + ((size_t)jt * A.cfg.nA + fa) * tri(n);
                    if (!(__ldg(src) == __ldg(src))) return;   // not positive definite: normal path
                    full_set_start(lam0);
                    for (int i = lane; i < tri(n); i += 32) S[W.T + i] = __ldg(src + i);
                    __syncwarp();
                    t_ready = true;
                };
                // Brent methods (X2, GCV, BayesReg): the reference re-solves at the returned lambda = Brent's best
                // abscissa xf, a point that was already evaluated.  The solution of that evaluation is kept in the
                // (otherwise unused) L-curve arrays whenever xf moves, and handed out at the end instead of one more
                // NNLS solve (same minimiser; MET2_T2_FLAG_COLD_START keeps the reference's extra solve).
                int p_snap = 0;
                double sse_snap = 0.0;
                const int oSx = oLx, oSi = oLx + 32 * NS;   // x [32 NS doubles], ix [32 NS ints]
                auto snapshot = [&](double sse_now) {
#pragma unroll
                    for (int tt = 0; tt < NS; ++tt) {
                        const int i = lane + 32 * tt;
                        if (i < p) {
                            S[oSx + i] = S[W.xs + i];
                            SI(oSi, i) = SI(W.ix, i);
                        }
                    }
                    p_snap = p;
                    sse_snap = sse_now;
                };
                auto restore = [&]() {
                    __syncwarp();
#pragma unroll
                    for (int sidx = 0; sidx < NS; ++sidx) {
                        const int col = NS * lane + sidx;
                        if (col < n) S[W.xc + col] = 0.0;
                    }
                    __syncwarp();
#pragma unroll
                    for (int tt = 0; tt < NS; ++tt) {
                        const int i = lane + 32 * tt;
                        if (i < p_snap) {
                            const int ci = SI(oSi, i);
                            const double xv = S[oSx + i];
                            S[W.xs + i] = xv;
                            SI(W.ix, i) = ci;
                            S[W.xc + ci] = xv;
                        }
                    }
                    p = p_snap;
                    __syncwarp();
                    (void)fit_and_sse<NS, ME>(W, Dt, oM, m, p, lane, fit);
                };
                while (true) {
                    // every solve after the first starts from the previous solution (support + coefficients)
                    p = nnls_gram<NS, GSH, PS>(W, oG, Gg, ldg, oKb, reg, lam, n, reg ? m + n : m, lane, nst,
                                            warm ? p : 0, t_ready);
                    t_ready = false;
                    if (method == MET2_REG_NNLS && nst == 0 && p > 0)
                        refine_on_support<NS, ME>(W, Dt, oM, m, p, lane, false, 0.0, oKb, n);
                    if (method == MET2_REG_BAYESREG && reg && nst == 0 && p > 0)
                        refine_on_support<NS, ME>(W, Dt, oM, m, p, lane, true, lam, oKb, n);
                    const double sse = fit_and_sse<NS, ME>(W, Dt, oM, m, p, lane, fit);
                    if (stage == ST_FINAL) {
                        if (method == MET2_REG_GCV && (A.cfg.flags & MET2_T2_FLAG_GCV_EVAL)) {
                            const double nrm = reg_norm2<NS>(W, oLb, n, lane);
                            int kept = 0;
                            regv = gcv_cost<NS, GSH>(W, oG, Gg, ldg, oLb, n, m, lane, lam, sse, nrm, p, kept);
                            st |= ((unsigned)kept & 0xffu) << 16;     // MET2_T2_FLAG_GCV_EVAL: kept rank in bits 16-23
                            (void)fit_and_sse<NS, ME>(W, Dt, oM, m, p, lane, fit);
                        } else
                        if (method == MET2_REG_X2 && !(A.cfg.flags & MET2_T2_FLAG_REG_IS_LAMBDA))
                            regv = sse / SSE;   // k_est is what the orchestrator stores (motor...:141-143)
                        else
                            regv = lam;         // NNLS -> 0
                        break;
                    }
                    if (method == MET2_REG_GCV) {
                        // algorithms.py:276-296
                        const double nrm = reg_norm2<NS>(W, oLb, n, lane);
                        int kept = 0;
                        const double cost = gcv_cost<NS, GSH>(W, oG, Gg, ldg, oLb, n, m, lane, lam, sse, nrm, p, kept);
                        if (A.cfg.flags & MET2_T2_FLAG_GCV_GRID) {
                            // np.argmin over the grid: first minimum, a NaN wins and stays
                            if (gi == 0 || (SSE == SSE && (cost < SSE || cost != cost))) {
                                SSE = cost;      // best objective so far (SSE is unused by GCV otherwise)
                                beta = lam;      // ... and its lambda
                            }
                            ++gi;
                            if (gi < A.cfg.nLambda) {
                                lam = S[oLam + gi];
                            } else {
                                lam = beta;
                                stage = ST_FINAL;
                            }
                        } else {
                            const double lam_eval = lam;
                            const bool more = B.feed(cost, lam);
                            if (warm && B.xf == lam_eval) snapshot(sse);
                            if (!more) {
                                lam = B.xf;
                                stage = ST_FINAL;
                                if (warm) {
                                    restore();
                                    regv = lam;
                                    break;
                                }
                            }
                        }
                    } else if (method == MET2_REG_BAYESREG) {
                        // bayesian_interpolation.py:84-105
                        if (stage == ST_PLAIN0) {
                            int nnz = 0;
#pragma unroll
                            for (int tt = 0; tt < NS; ++tt) {
                                int i = lane + 32 * tt;
                                if (i < p && S[W.xs + i] > 0.0) ++nnz;
                            }
                            nnz = __reduce_add_sync(FULL_MASK, nnz);
                            const double dof = fmax((double)(m - nnz), 1.0);
                            const double sigma = sqrt(sse / dof);
                            beta = 1.0 / (sigma * sigma);
                            lam = B.start(A.cfg.brent_lo, A.cfg.brent_hi, A.cfg.brent_xatol, A.cfg.maxfun);
                            reg = true;
                            stage = ST_SEARCH;
                        } else {
                            const double nrm = reg_norm2<NS>(W, oLb, n, lane);
                            const double* ttab = nullptr;
                            if (A.tfull) {
                                for (int q = 0; q < A.ntab; ++q)
                                    if (lam == __ldg(A.lam_tab + q)) ttab = A.tfull + ((size_t)q * A.cfg.nA + fa) * tri(n);
                                if (ttab && !(__ldg(ttab) == __ldg(ttab))) ttab = nullptr;   // not positive definite
                            }
                            const double cost = bayes_cost<NS, GSH>(W, oG, Gg, ldg, oKb, n, m, lane, lam, beta, sse, nrm,
                                                               A.cfg.log_det_L, st, ttab);
                            const double lam_eval = lam;
                            const bool more = B.feed(cost, lam);
                            if (warm && B.xf == lam_eval) snapshot(sse);
                            if (!more) {
                                lam = B.xf;
                                stage = ST_FINAL;
                                if (warm) {
                                    restore();
                                    regv = lam;
                                    break;
                                }
                            }
                        }
                    } else if (method == MET2_REG_X2) {
                        if (stage == ST_PLAIN0) {
                            SSE = sse;
                            if (SSE == 0.0) st |= MET2_ST_SSE_ZERO;
                            lam = B.start(A.cfg.brent_lo, A.cfg.brent_hi, A.cfg.brent_xatol, A.cfg.maxfun);
                            reg = true;
                            stage = ST_SEARCH;
                            if (warm && (A.cfg.flags & MET2_T2_FLAG_FULL_START) && lam >= 1.0) {
                                try_table(lam);
                                if (!t_ready) full_set_start(lam);
                            }
                        } else {
                            const double cost = fabs(sse - A.cfg.factor * SSE) / SSE;
                            const double lam_eval = lam;
                            const bool more = B.feed(cost, lam);
                            if (warm && B.xf == lam_eval) snapshot(sse);
                            if (more && (A.cfg.flags & MET2_T2_FLAG_FULL_START)) try_table(lam);
                            if (!more) {
                                lam = B.xf;
                                stage = ST_FINAL;
                                if (warm) {
                                    restore();
                                    // k_est is what the orchestrator stores (motor...:141-143)
                                    regv = (A.cfg.flags & MET2_T2_FLAG_REG_IS_LAMBDA) ? lam : sse_snap / SSE;
                                    break;
                                }
                            }
                        }
                    } else {   // L-curve grid
                        const double nrm = reg_norm2<NS>(W, oLb, n, lane);
                        if (lane == 0) {
                            S[oLx + gi] = log(sse + 1e-200);
                            S[oLy + gi] = log(nrm + 1e-200);
                        }
                        __syncwarp();
                        ++gi;
                        if (gi < A.cfg.nLambda) {
                            lam = S[oLam + gi];
                        } else {
                            lam = S[oLam + select_corner_warp(oLx, oLy, A.cfg.nLambda, lane)];
                            stage = ST_FINAL;
                        }
                    }
                }
                if (nst) st |= MET2_ST_ITMAX;
            }
            // ---- outputs: fsol = x*km, Est_Signal = (D x)*km, reg, maps (motor...:153-155, 443-472)
            const bool fitted = !(st & MET2_ST_SKIPPED);
            const double kmo = fitted ? km : 0.0;
            double xk[NS];
            double vt = 0.0;
#pragma unroll
            for (int sidx = 0; sidx < NS; ++sidx) {
                int col = NS * lane + sidx;
                xk[sidx] = (col < n && fitted) ? S[W.xc + col] * kmo : 0.0;
                vt += xk[sidx];
                if (col < n) A.fsol[v * n + col] = xk[sidx];
            }
#pragma unroll
            for (int u = 0; u < ME; ++u) {
                int e = lane + 32 * u;
                if (e < m) A.est[v * m + e] = fitted ? fit[u] * kmo : 0.0;
            }
            vt = warp_sum(vt) + 1.0e-16;
            double sm = 0.0, stt = 0.0, sc = 0.0, lm = 0.0, lt = 0.0;
#pragma unroll
            for (int sidx = 0; sidx < NS; ++sidx) {
                int col = NS * lane + sidx;
                if (col < n) {
                    double xn = xk[sidx] / vt;
                    unsigned char cm = scomp[col];
                    if (cm & 1) {
                        sm += xn;
                        lm += xn * S[oLogT2 + col];
                    }
                    if (cm & 2) {
                        stt += xn;
                        lt += xn * S[oLogT2 + col];
                    }
                    if (cm & 4) sc += xn;
                }
            }
            sm = warp_sum(sm);
            stt = warp_sum(stt);
            sc = warp_sum(sc);
            lm = warp_sum(lm);
            lt = warp_sum(lt);
            if (lane == 0) {
                double* mp = A.maps + v * 6;
                mp[0] = sm;
                mp[1] = stt;
                mp[2] = sc;
                mp[3] = exp(lm / (sm + 1.0e-16));
                mp[4] = exp(lt / (stt + 1.0e-16));
                mp[5] = vt;
                A.reg[v] = fitted ? regv : 0.0;
                A.status[v] = st;
            }
            __syncwarp();
        }
    }
}

struct T2Geom {
    int grid, warps, pmax, max_tiles;
    int tile_big, tile_small, switch_off;
    size_t smem;
};

template <int NS>
static inline T2Geom t2_geometry(long long V, const met2_t2_cfg* cfg, const Overrides& ov) {
    T2Geom g;
    const int n = cfg->nT2, m = cfg->nTE;
    const bool plain = (cfg->method == MET2_REG_NNLS);
    g.pmax = plain ? (n < m ? n : m) : n;
    if (cfg->method == MET2_REG_GCV)   // the T region also hosts the GCV workspace (C: n x 21, H: 20 x 21)
        while (tri(g.pmax) < gcv_region_doubles(n)) ++g.pmax;
    size_t tables = sizeof(double) * (size_t)t2_table_doubles(n, t2_gram_in_shared(NS));
    size_t per_warp = sizeof(double) * (size_t)t2_warp_doubles<NS>(g.pmax);
    size_t budget = 227 * 1024 - 1024;
    int warps = (int)((budget - tables) / per_warp);
    if (warps > T2_MAX_THREADS / 32) warps = T2_MAX_THREADS / 32;
    if (warps < 1) warps = 1;
    if (ov.t2_warps >= 1 && ov.t2_warps < warps) warps = ov.t2_warps;
    g.warps = warps;
    g.smem = tables + per_warp * warps;
    int per_sm = (int)(budget / (g.smem + 1024));
    if (per_sm < 1) per_sm = 1;
    int sms = sm_count();
    if (sms <= 0) sms = 148;
    g.grid = sms * per_sm;
    // guided self-scheduling of the tile list (t2_tiles_kernel): ~8 large tiles per CTA, then small tiles for the last
    // ~12 % of the voxels; MET2_T2_TILE=<n> forces a uniform tile size
    long long big = V / ((long long)g.grid * 8);
    big = (big + 31) & ~31LL;
    if (big < 64) big = 64;
    if (big > T2_TILE_MAX) big = T2_TILE_MAX;
    g.tile_big = (int)big;
    g.tile_small = T2_TILE_MIN;
    g.switch_off = (int)(V - V / 8);
    if (ov.t2_tile >= 1) {
        g.tile_big = g.tile_small = ov.t2_tile;
        g.switch_off = (int)V;
    }
    g.max_tiles = (int)(V / g.tile_small) + cfg->nA + 1;
    return g;
}

static inline T2Geom t2_geometry_any(long long V, const met2_t2_cfg* cfg, const Overrides& ov) {
    int ns = (cfg->nT2 + 31) / 32;
    if (ns <= 2) return t2_geometry<2>(V, cfg, ov);
    if (ns == 3) return t2_geometry<3>(V, cfg, ov);
    return t2_geometry<4>(V, cfg, ov);
}

template <int NS, int ME, int METHOD>
static int t2_launch_one(const T2Args& A, const T2Geom& g, cudaStream_t st) {
    cudaError_t e = cudaFuncSetAttribute(t2_fit_kernel<NS, ME, METHOD>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)g.smem);
    if (e != cudaSuccess) return set_error(MET2_ERR_CUDA, "t2_fit attr (%zu B): %s", g.smem, cudaGetErrorString(e));
    MET2_LAUNCH(g.grid, g.warps * 32, g.smem, st, t2_fit_kernel<NS, ME, METHOD>)(A);
    count_launch();
    return check_launch("t2_fit_kernel");
}

template <int METHOD>
static int t2_launch_method(const T2Args& A, const T2Geom& g, cudaStream_t st) {
    const int ns = (A.cfg.nT2 + 31) / 32, me = (A.cfg.nTE + 31) / 32;
    if (ns <= 2 && me == 1) return t2_launch_one<2, 1, METHOD>(A, g, st);
    if (ns <= 2 && me == 2) return t2_launch_one<2, 2, METHOD>(A, g, st);
    if (ns == 3 && me == 1) return t2_launch_one<3, 1, METHOD>(A, g, st);
    if (ns == 3 && me == 2) return t2_launch_one<3, 2, METHOD>(A, g, st);
    if (ns == 4 && me == 1) return t2_launch_one<4, 1, METHOD>(A, g, st);
    if (ns == 4 && me == 2) return t2_launch_one<4, 2, METHOD>(A, g, st);
    return set_error(MET2_ERR_UNSUPPORTED, "met2_t2_fit: unsupported template sizes");
}

// one definition per method, in met2_t2_m<method>.cu
int t2_launch_nnls(const T2Args& A, const T2Geom& g, cudaStream_t st);
int t2_launch_t2sparc(const T2Args& A, const T2Geom& g, cudaStream_t st);
int t2_launch_x2(const T2Args& A, const T2Geom& g, cudaStream_t st);
int t2_launch_lcurve(const T2Args& A, const T2Geom& g, cudaStream_t st);
int t2_launch_bayesreg(const T2Args& A, const T2Geom& g, cudaStream_t st);
int t2_launch_gcv(const T2Args& A, const T2Geom& g, cudaStream_t st);
// met2_t2_echo_r16.cu / met2_t2_echo_r24.cu (MET2_T2_FLAG_ECHO_SPACE; rank = cfg.echo_rank)
bool t2_echo_eligible(const met2_t2_cfg* cfg);
int t2_launch_echo_r16(const T2Args& A, const Overrides& ov, cudaStream_t st);
int t2_launch_echo_r24(const T2Args& A, const Overrides& ov, cudaStream_t st);
// met2_t2_echo_reg_r16.cu / met2_t2_echo_reg_r24.cu (L-curve and BayesReg in the reduced echo space)
int t2_launch_echo_reg_r16(const T2Args& A, const Overrides& ov, cudaStream_t st);
int t2_launch_echo_reg_r24(const T2Args& A, const Overrides& ov, cudaStream_t st);

}  // namespace met2
