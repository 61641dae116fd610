// met2_t2_echo_impl.cuh — Tikhonov NNLS in REDUCED ECHO SPACE for a diagonal regularisation matrix (reg_matrix I and InvT2):
// the X2 search (algorithms.py:211-233) and the fixed-lambda solve of T2SPARC (algorithms.py:262-269, motor...:138).
// Selected with MET2_T2_FLAG_ECHO_SPACE; batched.Met2Plan sets the flag whenever the configuration is eligible.
//
// For L = diag(l) and lam > 0 the Tikhonov problem
//     min_{x >= 0} |D x - b|^2 + lam |L x|^2,      Dt = D diag(1/l),  xt = l * x  (same sign pattern)
// has, on a positive set P, the stationary point (push-through identity)
//     v = (lam I + M_P)^-1 b,   M_P = sum_{j in P} dt_j dt_j^T   (independent of lam)
//     zt_P = Dt_P^T v,          w_Z = lam Dt_Z^T v               (r = b - Dt_P zt_P = lam v)
// so ONE product g = Dt^T v gives the coefficients on P and the dual on Z, a column entering / leaving P is a rank-one
// change of M_P, and a new lambda costs one factorisation of an echo-space matrix instead of a p x p one (p up to 60).
// With lam > 0 both acceptance tests of nnls.f pass identically (a regularised column is never dependent; its entering
// coefficient is w_j / (lam (1 + dt_j^T A^-1 dt_j)) > 0), so the control flow is the main loop + the interpolation loop
// of Lawson-Hanson (algorithms.py:55-82 -> nnls.f).
//
// REDUCED: the dictionary of one flip angle is numerically of rank ~20 (met2_basis.cu): D = U C with U: nTE x RD
// orthonormal, C = U^T D: RD x nT2 (RD = 24), exact to the rounding of D's own entries.  Every quantity above then
// lives in RD dimensions — b -> bt = U^T b, Dt -> Ct = C diag(1/l), M_P = Ct_P Ct_P^T (24 x 24) — and the part of b
// outside range(U) only adds the constant |b - U bt|^2 to every residual.  Against the unreduced echo-space kernel of
// round 2's first GPU call (32 x 32 factors): tri(24) = 300 instead of 528 doubles per factor, 3 instead of 4 diagonal
// blocks per refactorisation, 24- instead of 32-step triangular products, and nTE no longer limited to 32.  CPU
// prototype against voxels fitted by the unmodified reference (tools/proto_reduced_echo.py): 0 of 300 support
// disagreements, spectra within 1.1e-12 (RD = 24 and 20; the Gram-domain kernel: 1.4e-9).
//
// The factor is the upper-triangular inverse Cholesky factor T, A^-1 = T T^T, A = lam I + M_P:
//   new lambda     : rebuild_T_blocked (the FP64-tensor-core blocked factorisation of met2_nnls.cuh) on M_P + lam I
//   A' = A + s d d^T: u = T^T d;  (I + s u u^T)^-1 = Q Q^T with Q upper triangular, Q_jj = delta_j, Q_ij = u_i q_j (i < j);
//                    with tau_k = sum_{j <= k} u_j^2 (one warp scan), h_k = 1 + s tau_k:
//                        delta_k = sqrt(h_{k-1} / h_k),   q_k = -s u_k / (h_k delta_k)
//                    T' = T Q is a running sum along each ROW of T (one row per lane):
//                        T'[r][j] = delta_j T[r][j] + q_j acc,   acc += T[r][j] u_j
//                    (s = +1: h >= 1, no cancellation; s = -1: h_k >= 1 - u.u > 0, rebuilt from M_P if that fails).
// The plain NNLS of X2 (lam = 0: the SSE of algorithms.py:213-214) stays in the Gram domain (nnls_gram), with its
// right-hand side, residual and D-space candidate test taken in the same reduced space.
//
// Compiled once per rank of the reduced space (met2_t2_echo_r16.cu, met2_t2_echo_r24.cu define MET2_ECHO_RD, a namespace
// and the name of the launcher): RD = 16 whenever the rank-16 reduction leaves a residual below 4e-12 (the reference's
// 32-echo protocol: 1.6e-12, sigma_17 / sigma_1 = 6e-13; measured on 20 480 voxels fitted by the unmodified reference: 0
// active-set disagreements, spectra within 7.8e-9 — the accuracy class of the Gram-domain kernels — and 19 % less time
// than RD = 24: two DMMA blocks per refactorisation instead of three, 16-step triangular products), RD = 24 otherwise
// (exact to the rounding of the dictionary's entries: 1e-16).
#include "met2_t2_impl.cuh"

#if !defined(MET2_ECHO_RD) || !defined(MET2_ECHO_NS) || !defined(MET2_ECHO_LAUNCH)
#error "met2_t2_echo_impl.cuh is included by met2_t2_echo_r<rank>.cu, which define MET2_ECHO_RD / _NS / _LAUNCH"
#endif
// MET2_ECHO_PART 1 (default): the X2 / T2SPARC kernels of this file; 2: the L-curve / BayesReg kernel of
// met2_t2_echo_reg_impl.cuh (met2_t2_echo_reg_r<rank>.cu) on the same device functions — separate translation units so
// that they compile in parallel.
#ifndef MET2_ECHO_PART
#define MET2_ECHO_PART 1
#endif

namespace met2 {
namespace MET2_ECHO_NS {

constexpr int RD = MET2_ECHO_RD;      // rows of the reduced system (DMMA blocks of 8)
constexpr int EC_LDD = RD + 2;        // row stride of the staged Ct table [column][row]: even (16-byte rows for 128-bit
                                      // loads with lane = column: a quarter warp covers all 32 banks) and conflict-free
                                      // for lane = row
constexpr int EC_NCOL = 64;           // columns of the X2 kernel (nT2 <= 64), zero rows beyond nT2

struct EchoOff {
    int Ct, RC, Mp, B, V, D;   // offsets into S: staged Ct table, (row, column) bytes of the packed triangle; per warp:
                               // M_P packed lower, bt (RD), v (RD), d (RD)
};
constexpr int EC_RC_DOUBLES = (2 * tri(RD) + 7) / 8;   // tri(RD) byte pairs

// (row, column) of every packed lower-triangle entry, as bytes: rc[2 e] = r, rc[2 e + 1] = c for e = tri(r) + c.
__device__ __forceinline__ void echo_stage_rc(int oRC) {
    unsigned char* rc = reinterpret_cast<unsigned char*>(S + oRC);
    for (int e = threadIdx.x; e < tri(RD); e += blockDim.x) {
        int r = 0;
        while (tri(r + 1) <= e) ++r;
        rc[2 * e] = (unsigned char)r;
        rc[2 * e + 1] = (unsigned char)(e - tri(r));
    }
}

// per-warp shared memory of the X2 kernel (doubles): Slots<2>(pmax RD) | M_P packed lower tri(RD) | raw signal, later
// the Brent-best snapshot of xt (64) | bt (RD) | v (RD) | d (RD) — 8.8 KB, so that 20 warps fit beside the tables
// (the kernel is latency bound: 8 / 12 / 14 / 16 warps measured 329 / 250 / 234 / 211 ms per volume)
__host__ __device__ __forceinline__ int echo_warp_doubles() {
    return (Slots<2>::doubles(RD) + tri(RD) + 64 + 3 * RD + 7) & ~7;
}
// CTA tables (doubles): G [n][ldg] | Ct [64][EC_LDD] | U [m][RD] | M_full packed tri(RD) | l (64) | 1/l (64) | logT2 (64) |
// comp (8) | (row, column) bytes of the packed triangle
__host__ __device__ __forceinline__ int echo_table_doubles(int n, int m) {
    return (n * t2_ldg(n) + EC_NCOL * EC_LDD + m * RD + tri(RD) + 3 * 64 + 8 + EC_RC_DOUBLES + 31) & ~31;
}

// unrolled, compile-time-indexed inner products and factor update in the X2 / T2SPARC kernels only (see echo_tmul
// below); the unrolled update in the L-curve / BayesReg kernel measured slower (L-curve 296 -> 319 ms, BayesReg 340 -> 350)
constexpr bool ECHO_UNROLLED_TRI = (MET2_ECHO_PART == 1);

// g = Ct^T v for v at S[oV .. oV + RD): lane + 32 s = column (NC column slots per lane: nT2 <= 32 NC).
template <int NC>
__device__ __forceinline__ void echo_gprod(const EchoOff& O, int oV, int lane, double (&g)[NC]) {
    double g0[NC], g1[NC];
#pragma unroll
    for (int s = 0; s < NC; ++s) g0[s] = g1[s] = 0.0;
    const int r0 = O.Ct + lane * EC_LDD;
#pragma unroll (ECHO_UNROLLED_TRI ? RD / 2 : 1)
    for (int e = 0; e < RD; e += 2) {
        double vv[2];
        lds_vec<2>(oV + e, vv);
#pragma unroll
        for (int s = 0; s < NC; ++s) {
            double dd[2];
            lds_vec<2>(r0 + 32 * s * EC_LDD + e, dd);
            g0[s] = fma(dd[0], vv[0], g0[s]);
            g1[s] = fma(dd[1], vv[1], g1[s]);
        }
    }
#pragma unroll
    for (int s = 0; s < NC; ++s) g[s] = g0[s] + g1[s];
}

// The two triangular products of the RD x RD factor with compile-time triangle offsets and 128-bit broadcast loads of the
// vector (S[oV ..], oV even: every per-warp region starts on an even offset and tri(16), tri(24), 64 and RD are even).
// Same association as tmul / tmul_transposed of met2_nnls.cuh (even columns in one accumulator, odd in the other), so the
// results are bitwise the same; those keep a runtime trip count and per-iteration triangle arithmetic because they serve
// any p — here they were 17 % of the X2 kernel's instructions.  Measured (GPU call 24, config-2 volume): X2-I 136.5 ->
// 131.1 ms, T2SPARC 51.3 -> 49.9 ms; but the L-curve / BayesReg kernel, which is bound by instruction fetch, lost what
// the +128 SASS instructions per call site cost (L-curve 293 -> 323 ms, BayesReg 339 -> 346 ms): MET2_ECHO_PART 2 keeps
// the compact generic products.  Unrolling further does not pay either: the seven steps of the 8 x 8 diagonal-block
// elimination and the M_P update with compile-time offsets (+ 976 SASS instructions) took X2-I from 128 to 166 ms
// (GPU call 27) — the kernel sits at the edge of what the instruction caches hold.
// out_r = sum_{c >= r} T(r, c) v_c  (lane = row r; lanes >= RD get 0)
__device__ __forceinline__ double echo_tmul(int oT, int oV, int lane) {
    if (!ECHO_UNROLLED_TRI) {
        double v[1];
        tmul<1>(oT, oV, RD, lane, v);
        return v[0];
    }
    double a0 = 0.0, a1 = 0.0;
#pragma unroll
    for (int c = 0; c < RD; c += 2) {
        double vv[2];
        lds_vec<2>(oV + c, vv);
        const double e0 = (lane <= c) ? S[oT + tri(c) + lane] : 0.0;
        const double e1 = (lane <= c + 1) ? S[oT + tri(c + 1) + lane] : 0.0;
        a0 = fma(e0, vv[0], a0);
        a1 = fma(e1, vv[1], a1);
    }
    return a0 + a1;
}
// out_i = sum_{k <= i} T(k, i) v_k  (lane = column i; lanes >= RD get 0)
__device__ __forceinline__ double echo_tmul_t(int oT, int oV, int lane) {
    if (!ECHO_UNROLLED_TRI) {
        double v[1];
        tmul_transposed<1>(oT, oV, RD, lane, v);
        return v[0];
    }
    const int base = oT + tri(lane);
    const int kmax = (lane < RD) ? lane : -1;
    double a0 = 0.0, a1 = 0.0;
#pragma unroll
    for (int k = 0; k < RD; k += 2) {
        double vv[2];
        lds_vec<2>(oV + k, vv);
        const double t0 = (k <= kmax) ? S[base + k] : 0.0;
        const double t1 = (k + 1 <= kmax) ? S[base + k + 1] : 0.0;
        a0 = fma(t0, vv[0], a0);
        a1 = fma(t1, vv[1], a1);
    }
    return a0 + a1;
}

// v = T (T^T bt), g = Ct^T v.  lane = position / row for the triangular products.
template <int NC, int NS>
__device__ __forceinline__ void echo_solve(const Slots<NS>& W, const EchoOff& O, int lane, double (&g)[NC], double& y,
                                           bool& y_ok) {
    // y = T^T bt: fresh after a refactorisation, otherwise carried through the rank-one updates (echo_change)
    if (!y_ok) {
        y = echo_tmul_t(W.T, O.B, lane);
        y_ok = true;
    }
    if (lane < RD) S[W.rs + lane] = y;
    __syncwarp();
    const double v = echo_tmul(W.T, W.rs, lane);
    if (lane < RD) S[O.V + lane] = v;
    __syncwarp();
    echo_gprod<NC>(O, O.V, lane, g);
    __syncwarp();
}

// T <- inverse Cholesky factor of M_P + lam I.  Returns false if a pivot is not positive.
template <int NS>
__device__ __forceinline__ bool echo_refactor(const Slots<NS>& W, const EchoOff& O, double lam, int lane) {
    auto Aent = [&](int r, int c) -> double {
        const int hi = (r > c) ? r : c, lo = (r > c) ? c : r;
        double a = S[O.Mp + tri(hi) + lo];
        if (r == c) a += lam;
        return a;
    };
    __syncwarp();
    return rebuild_T_blocked<NS>(W, Aent, RD, lane);
}

// M_P += sgn d d^T on the packed lower triangle, d = column j of the staged Ct table; leaves d in S[O.D..].
// The tri(RD) = 300 packed entries are dealt to the 32 lanes (entry e = lane + 32 t) with their (row, column) read from
// a byte table built once per CTA (O.RC): ten balanced steps instead of RD steps of a half-empty warp (the row-per-lane
// version was the single hottest line of the first reduced kernel, 7.6 % of its instructions).
__device__ __forceinline__ void echo_mp_rank1(const EchoOff& O, int j, double sgn, int lane) {
    const double d = (lane < RD) ? S[O.Ct + j * EC_LDD + lane] : 0.0;
    __syncwarp();
    if (lane < RD) S[O.D + lane] = d;
    __syncwarp();
    const unsigned char* rc = reinterpret_cast<const unsigned char*>(S + O.RC);
#pragma unroll 1
    for (int e = lane; e < tri(RD); e += 32) {
        const double dr = S[O.D + rc[2 * e]], dc = S[O.D + rc[2 * e + 1]];
        S[O.Mp + e] = fma(sgn * dr, dc, S[O.Mp + e]);
    }
    __syncwarp();
}

// The update of T that goes with M_P += sgn d d^T (echo_mp_rank1 has left d in S[O.D..]): T' = T Q, and y' = Q^T y when y
// is valid.  Returns false — T untouched — if the downdate lost positivity in floating point; the caller then
// refactors from the (already updated) M_P.
template <int NS>
__device__ __forceinline__ bool echo_update_T(const Slots<NS>& W, const EchoOff& O, double sgn, int lane, double& y,
                                              bool y_ok) {
    // ---- u = T^T d, prefix sums of u^2
    const double u[1] = {echo_tmul_t(W.T, O.D, lane)};
    double tau[1] = {u[0] * u[0]};
    warp_scan_positions<1>(tau, lane);
    const double h = fma(sgn, tau[0], 1.0);
    double hm1 = __shfl_up_sync(FULL_MASK, h, 1);
    if (lane == 0) hm1 = 1.0;
    const bool okh = (h > 0.0) && (hm1 > 0.0);
    if (!__all_sync(FULL_MASK, okh)) return false;
    const double delta = sqrt(hm1 / h);
    const double q = -sgn * u[0] / (h * delta);
    if (y_ok) {
        // y' = Q^T y:  y'_j = delta_j y_j + q_j sum_{i < j} u_i y_i   (one more scan instead of a fresh T'^T b)
        double e[1] = {u[0] * y};
        const double own = e[0];
        warp_scan_positions<1>(e, lane);
        y = fma(q, e[0] - own, delta * y);
    }
    if (lane < RD) {
        S[W.gs + lane] = delta;
        S[W.gs + 32 + lane] = q;
        S[W.rs + lane] = u[0];
    }
    __syncwarp();
    // ---- T' = T Q, one row of T per lane (row r has entries in columns j >= r)
    if (ECHO_UNROLLED_TRI) {
        // compile-time column index: constant triangle offsets, (delta, q, u) of two columns per 128-bit broadcast load
        double acc = 0.0;
#pragma unroll
        for (int c = 0; c < RD; c += 2) {
            double dl[2], qq[2], uu[2];
            lds_vec<2>(W.gs + c, dl);
            lds_vec<2>(W.gs + 32 + c, qq);
            lds_vec<2>(W.rs + c, uu);
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                if (lane <= c + h) {
                    const int a = W.T + tri(c + h) + lane;
                    const double t = S[a];
                    S[a] = fma(dl[h], t, qq[h] * acc);
                    acc = fma(t, uu[h], acc);
                }
            }
        }
    } else if (lane < RD) {
        double acc = 0.0;
#pragma unroll 1
        for (int c = lane; c < RD; ++c) {
            const int a = W.T + tri(c) + lane;
            const double t = S[a];
            S[a] = fma(S[W.gs + c], t, S[W.gs + 32 + c] * acc);
            acc = fma(t, S[W.rs + c], acc);
        }
    }
    __syncwarp();
    return true;
}

// Lawson-Hanson in echo space for one lambda.  On entry M_P belongs to the set `inP` (bit s of lane l = column l + 32 s)
// and x[s] holds a feasible point on it (x > 0 on P, 0 elsewhere); an empty set is allowed.  refactor: T has to be
// rebuilt from M_P + lam I first (a new lambda); otherwise T is the factor for `inP` already.
// block_drop: the entry set is the FULL column set — drop every column whose unconstrained coefficient is not positive
// in one go before the usual interpolation loop (x stays feasible on the reduced set).
// On exit inP / x hold the solution (scaled unknowns xt = l * x); status bit 0: itmax, bit 1: a pivot was not positive.
//
// One loop with ONE inlined site each for the refactorisation, the rank-one change and the solve (the version with
// nnls.f's two nested loops inlined the solve and the change twice and the blocked refactorisation three times: the
// kernels are instruction-fetch bound, DESIGN.md §6): A. apply the pending set changes — the entering column or the
// leaving ones, lowest column first; B. solve; C. `secondary`: the feasibility test / interpolation step of nnls.f's
// inner loop; D. otherwise: the entering column, arg-max of the dual over the zero set (outer loop).
template <int NC, int NS>
__device__ __forceinline__ void echo_nnls(const Slots<NS>& W, const EchoOff& O, int n, double lam, int lane,
                                          unsigned& inP, double (&x)[NC], int& status, bool block_drop, bool refactor) {
    const int itmax = 3 * n;
    int iter = 0;
    bool secondary = __any_sync(FULL_MASK, inP != 0u);   // a non-empty entry set is checked for feasibility first
    double g[NC];
    double y = 0.0;        // y = T^T bt of the current factor (lane = position), valid when y_ok
    bool y_ok = false;
    int enter_j = -1;      // column that enters next
    unsigned outm = 0u;    // columns that leave next
    while (true) {
        // ---- A. pending set changes
        while (true) {
            int k;
            double sgn;
            if (enter_j >= 0) {
                k = enter_j;
                sgn = 1.0;
                enter_j = -1;
            } else {
                k = 0x7fffffff;
#pragma unroll
                for (int s = NC - 1; s >= 0; --s)
                    if ((outm >> s) & 1u) k = lane + 32 * s;
                k = (int)__reduce_min_sync(FULL_MASK, (unsigned)k);
                if (k == 0x7fffffff) break;
                sgn = -1.0;
                if ((k & 31) == lane) {
                    const unsigned bit = 1u << (k >> 5);
                    outm &= ~bit;
                    inP &= ~bit;
#pragma unroll
                    for (int s = 0; s < NC; ++s)
                        if (s == (k >> 5)) x[s] = 0.0;
                }
            }
            echo_mp_rank1(O, k, sgn, lane);
            // a downdate that loses positivity in floating point: T is rebuilt from the updated M_P below
            if (!refactor && !echo_update_T(W, O, sgn, lane, y, y_ok)) refactor = true;
        }
        if (refactor) {
            if (!echo_refactor(W, O, lam, lane)) status |= 2;
            refactor = false;
            y_ok = false;
        }
        // ---- B. solve for the current set
        if (secondary) {
            ++iter;
            if (iter > itmax) {
                status |= 1;
                break;
            }
        }
        echo_solve<NC>(W, O, lane, g, y, y_ok);
        // ---- C. feasibility on P (interpolation loop of nnls.f)
        if (secondary) {
            const bool drop_now = block_drop;
            block_drop = false;
            unsigned negm = 0u;
#pragma unroll
            for (int s = 0; s < NC; ++s)
                if (((inP >> s) & 1u) && g[s] <= 0.0) negm |= 1u << s;
            if (__any_sync(FULL_MASK, negm != 0u)) {
                if (drop_now) {
                    outm = negm;
                    continue;
                }
                double bt = 2.0;
                int bi = -1;
#pragma unroll
                for (int s = 0; s < NC; ++s) {
                    if ((negm >> s) & 1u) {
                        const double tt = x[s] / (x[s] - g[s]);
                        if (tt < bt) {
                            bt = tt;
                            bi = lane + 32 * s;
                        }
                    }
                }
                double alpha = 0.0;
                const int jb = warp_argmin_nonneg(bt, bi, alpha);
                if (jb < 0) {          // no step found: back to the outer loop with a fresh solve (nnls.f leaves the loop)
                    secondary = false;
                    continue;
                }
#pragma unroll
                for (int s = 0; s < NC; ++s) {
                    if ((inP >> s) & 1u) {
                        x[s] = x[s] + alpha * (g[s] - x[s]);
                        if (x[s] <= 0.0 || lane + 32 * s == jb) outm |= 1u << s;
                    }
                }
                continue;
            }
#pragma unroll
            for (int s = 0; s < NC; ++s) x[s] = ((inP >> s) & 1u) ? g[s] : 0.0;
            secondary = false;
        }
        // ---- D. entering column: arg-max of the dual w = lam g over the zero set (lam > 0: same order as g)
        if ((int)__reduce_add_sync(FULL_MASK, (unsigned)__popc(inP)) >= n) break;
        double bv = 0.0;
        int bj = -1;
#pragma unroll
        for (int s = 0; s < NC; ++s) {
            const int col = lane + 32 * s;
            if (col < n && !((inP >> s) & 1u) && g[s] > bv) {
                bv = g[s];
                bj = col;
            }
        }
        const int j = warp_argmax_pos(bv, bj);
        if (j < 0) break;
        if ((j & 31) == lane) inP |= 1u << (j >> 5);
        enter_j = j;
        secondary = true;
    }
}

// ft = Ct xt (reduced fit, lane = row; left in S[oF .. oF + RD) when oF >= 0) and |ft - bt|^2.  xt is read from
// S[oX + 0..n) (column space).
__device__ __forceinline__ double echo_fit_sse(int oX, const EchoOff& O, int n, int lane, int oF) {
    double f0 = 0.0, f1 = 0.0;
    if (lane < RD) {
        int j = 0;
#pragma unroll 1
        for (; j + 1 < n; j += 2) {
            f0 = fma(S[O.Ct + j * EC_LDD + lane], S[oX + j], f0);
            f1 = fma(S[O.Ct + (j + 1) * EC_LDD + lane], S[oX + j + 1], f1);
        }
        if (j < n) f0 = fma(S[O.Ct + j * EC_LDD + lane], S[oX + j], f0);
    }
    const double ft = f0 + f1;
    if (oF >= 0 && lane < RD) S[oF + lane] = ft;
    const double dd = (lane < RD) ? ft - S[O.B + lane] : 0.0;
    return warp_sum(dd * dd);
}

// Project the normalised signal S[oM .. oM + m) onto the reduced basis U ([m][RD] at S[oU..]): bt -> S[oB .. oB + RD),
// and return |b - U bt|^2, the part of every residual that no spectrum can reach.
template <int ME>
__device__ __forceinline__ double echo_project(int oU, int oM, int oB, int m, int lane) {
    double b0 = 0.0, b1 = 0.0;
    if (lane < RD) {
        int k = 0;
#pragma unroll 1
        for (; k + 1 < m; k += 2) {
            b0 = fma(S[oU + k * RD + lane], S[oM + k], b0);
            b1 = fma(S[oU + (k + 1) * RD + lane], S[oM + k + 1], b1);
        }
        if (k < m) b0 = fma(S[oU + k * RD + lane], S[oM + k], b0);
        S[oB + lane] = b0 + b1;
    }
    __syncwarp();
    double perp = 0.0;
#pragma unroll
    for (int u = 0; u < ME; ++u) {
        const int k = lane + 32 * u;
        if (k < m) {
            double a0 = 0.0, a1 = 0.0;
#pragma unroll 1
            for (int e = 0; e < RD; e += 2) {
                a0 = fma(S[oU + k * RD + e], S[oB + e], a0);
                a1 = fma(S[oU + k * RD + e + 1], S[oB + e + 1], a1);
            }
            const double r = S[oM + k] - (a0 + a1);
            perp = fma(r, r, perp);
        }
    }
    return warp_sum(perp);
}

// fit[u] (echo k = lane + 32 u) = sum_e U[k][e] ft[e] for ft at S[oF .. oF + RD): the fitted signal D x in echo space.
template <int ME>
__device__ __forceinline__ void echo_expand(int oU, int oF, int m, int lane, double (&fit)[ME]) {
#pragma unroll
    for (int u = 0; u < ME; ++u) {
        const int k = lane + 32 * u;
        double a0 = 0.0, a1 = 0.0;
        if (k < m) {
#pragma unroll 1
            for (int e = 0; e < RD; e += 2) {
                a0 = fma(S[oU + k * RD + e], S[oF + e], a0);
                a1 = fma(S[oU + k * RD + e + 1], S[oF + e + 1], a1);
            }
        }
        fit[u] = a0 + a1;
    }
}

// Outputs of one voxel (motor...:153-155, 443-472): fsol = x km, Est_Signal = (D x) km, reg, maps.  x in column space at
// S[oX .. oX + n), column = lane + 32 s.
template <int NC, int ME>
__device__ __forceinline__ void echo_outputs(const T2Args& A, long long v, int oX, int oLogT2, const unsigned char* scomp,
                                             int n, int m, int lane, unsigned st, double km, double regv,
                                             const double (&fit)[ME]) {
    const bool fitted = !(st & MET2_ST_SKIPPED);
    const double kmo = fitted ? km : 0.0;
    double xk[NC];
    double vt = 0.0;
#pragma unroll
    for (int s = 0; s < NC; ++s) {
        const int col = lane + 32 * s;
        xk[s] = (col < n && fitted) ? S[oX + col] * kmo : 0.0;
        vt += xk[s];
        if (col < n) A.fsol[v * n + col] = xk[s];
    }
#pragma unroll
    for (int u = 0; u < ME; ++u) {
        const int e = lane + 32 * u;
        if (e < m) A.est[v * m + e] = fitted ? fit[u] * kmo : 0.0;
    }
    vt = warp_sum(vt) + 1.0e-16;
    double sm = 0.0, stt = 0.0, sc = 0.0, lm = 0.0, lt = 0.0;
#pragma unroll
    for (int s = 0; s < NC; ++s) {
        const int col = lane + 32 * s;
        if (col < n) {
            const double xn = xk[s] / vt;
            const unsigned char cm = scomp[col];
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

// l = diag(L) from the row-band form (kband rows 5..9: kband[5 + d][r] = L[r][r + d - 2]); every other band must be 0.
__device__ __forceinline__ void echo_stage_diag(const T2Args& A, int ncol, int n, int oL, int oIL, int oLogT2,
                                                unsigned char* scomp, int* s_badL) {
    for (int i = threadIdx.x; i < ncol; i += blockDim.x) {
        double l = 1.0;
        if (i < n) {
            l = A.kband[7 * n + i];
            bool bad = !(l > 0.0) || !(l < 1e300);
            for (int d = 0; d < 5; ++d)
                if (d != 2 && A.kband[(5 + d) * n + i] != 0.0) bad = true;
            if (bad) atomicOr(s_badL, 1);
        }
        S[oL + i] = l;
        S[oIL + i] = 1.0 / l;
        S[oLogT2 + i] = (i < n) ? A.logT2[i] : 0.0;
        if (i < n) scomp[i] = A.comp[i];
    }
}

// Per-kernel launch bounds, measured on the config-2 volume (profiles/r02_ab_echo_warps.json; 640 / 768 / 896 / 1024
// threads = 20 / 24 / 28 / 30 warps per SM at 96 / 80 / 72 / 64 registers): X2 136.6 / 146.1 / 142.2 / 141.3 ms and the
// L-curve 293 / 344 / 363 / 394 ms are best at 640 (more resident warps sit in more phases of the kernel: instruction
// fetch), T2SPARC 56.8 / 54.6 / 52.3 / 51.4 ms and BayesReg (60 bins) 366 / 353 / 353 / 339 ms at 1024.
constexpr int ECHO_MAX_THREADS = 640;
constexpr int ECHO_TIK_MAX_THREADS = 1024;

static int echo_warps(size_t tables, size_t per_warp, const Overrides& ov, int max_threads = ECHO_MAX_THREADS) {
    const size_t budget = 227 * 1024 - 1024;
    int warps = tables < budget ? (int)((budget - tables) / per_warp) : 0;
    if (warps > max_threads / 32) warps = max_threads / 32;
    if (ov.t2_warps >= 1 && ov.t2_warps < warps) warps = ov.t2_warps;
    return warps;
}

#if MET2_ECHO_PART == 1

template <int ME>
__global__ void __launch_bounds__(ECHO_MAX_THREADS, 1) t2_echo_x2_kernel(T2Args A) {
    __shared__ int s_tile, s_next, s_badL;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int n = A.cfg.nT2, m = A.cfg.nTE;
    const int ldg = t2_ldg(n);
    const int oG = 0;
    const int oCt = oG + n * ldg;
    const int oU = oCt + EC_NCOL * EC_LDD;
    const int oMf = oU + m * RD;
    const int oL = oMf + tri(RD);
    const int oIL = oL + 64;
    const int oLogT2 = oIL + 64;
    unsigned char* scomp = reinterpret_cast<unsigned char*>(S + oLogT2 + 64);
    const int oRC = oLogT2 + 64 + 8;
    const int wbase = echo_table_doubles(n, m) + warp * echo_warp_doubles();
    Slots<2> W;
    W.carve(wbase, RD);
    EchoOff O;
    O.Ct = oCt;
    O.RC = oRC;
    O.Mp = wbase + Slots<2>::doubles(RD);
    const int oM = O.Mp + tri(RD);
    O.B = oM + 64;
    O.V = O.B + RD;
    O.D = O.V + RD;
    const int oSnap = oM;     // the raw signal is not needed once it is projected (bt) and km is in a register

    if (threadIdx.x == 0) s_badL = 0;
    __syncthreads();
    echo_stage_diag(A, 64, n, oL, oIL, oLogT2, scomp, &s_badL);
    echo_stage_rc(oRC);
    const int ntiles = A.counters[0];

    while (true) {
        __syncthreads();
        if (threadIdx.x == 0) {
            s_tile = atomicAdd(&A.counters[1], 1);
            s_next = 0;
        }
        __syncthreads();
        const int tile = s_tile;
        if (tile >= ntiles) break;
        const bool badL = (s_badL != 0);
        const int fa = A.tile_fa[tile];
        const int tstart = A.tile_start[tile], tcnt = A.tile_cnt[tile];
        const double* Cg = A.red_coef + (size_t)fa * n * RD;     // [n][RD]: C[e][j] at [j][e]
        {
            const double* Gg = A.G + (size_t)fa * n * n;
            for (int i = threadIdx.x; i < n * n; i += blockDim.x) {
                const int r = i / n;
                S[oG + r * ldg + (i - r * n)] = __ldg(Gg + i);
            }
            // Ct[j][e] = C[e][j] / l_j, zero rows beyond n and in the two pad columns
            for (int i = threadIdx.x; i < EC_NCOL * EC_LDD; i += blockDim.x) {
                const int j = i / EC_LDD, e = i - j * EC_LDD;
                S[oCt + i] = (j < n && e < RD) ? __ldg(Cg + j * RD + e) * S[oIL + j] : 0.0;
            }
            const double* Ug = A.red_basis + (size_t)fa * m * RD;
            for (int i = threadIdx.x; i < m * RD; i += blockDim.x) S[oU + i] = __ldg(Ug + i);
        }
        __syncthreads();
        // M_full = Ct-table product over ALL columns, packed lower triangle
        for (int i = threadIdx.x; i < tri(RD); i += blockDim.x) {
            int r = 0;
            while (tri(r + 1) <= i) ++r;
            const int c = i - tri(r);
            double a0 = 0.0, a1 = 0.0;
            int j = 0;
            for (; j + 1 < n; j += 2) {
                a0 = fma(S[oCt + j * EC_LDD + r], S[oCt + j * EC_LDD + c], a0);
                a1 = fma(S[oCt + (j + 1) * EC_LDD + r], S[oCt + (j + 1) * EC_LDD + c], a1);
            }
            if (j < n) a0 = fma(S[oCt + j * EC_LDD + r], S[oCt + j * EC_LDD + c], a0);
            S[oMf + i] = a0 + a1;
        }
        __syncthreads();

        while (true) {
            int it = 0;
            if (lane == 0) it = atomicAdd(&s_next, 1);
            it = __shfl_sync(FULL_MASK, it, 0);
            if (it >= tcnt) break;
            const long long v = A.perm[tstart + it];
            unsigned st = load_signal<ME>(A.sig, v, m, oM, lane);
            const int fav = A.fa_index[v];
            const bool normalise = !(A.cfg.flags & MET2_T2_FLAG_NO_NORMALISE);
            const double km = normalise ? S[oM] : 1.0;
            if (!st && (!(km > 0.0) || fav < 0 || fav >= A.cfg.nA)) st = MET2_ST_SKIPPED;
            if (!st && badL) st = MET2_ST_SKIPPED | MET2_ST_ECHO_BAD_L;
            double regv = 0.0;
            double fit[ME];
#pragma unroll
            for (int u = 0; u < ME; ++u) fit[u] = 0.0;
            if (!st) {
                __syncwarp();
#pragma unroll
                for (int u = 0; u < ME; ++u) {
                    const int e = lane + 32 * u;
                    if (e < m) S[oM + e] = S[oM + e] / km;
                }
                __syncwarp();
                const double perp = echo_project<ME>(oU, oM, O.B, m, lane);
                // ---- plain NNLS in the Gram domain -> SSE (algorithms.py:213-214): c = D^T b = l * (Ct^T bt)
                {
                    double g[2];
                    echo_gprod<2>(O, O.B, lane, g);
#pragma unroll
                    for (int s = 0; s < 2; ++s) {
                        const int j = lane + 32 * s;
                        if (j < n) S[W.cc + j] = g[s] * S[oL + j];
                    }
                    __syncwarp();
                }
                set_dspace<2>(W, Cg, O.B, lane);     // candidate test in the reduced space: rows of C, right-hand side bt
                int nst = 0;
                (void)nnls_gram<2, true, 1>(W, oG, nullptr, ldg, 0, false, 0.0, n, RD, lane, nst, 0, false);   // <= RD positions
                // xt0 = l * x0 -> column space; SSE = |Ct xt0 - bt|^2 + |b_perp|^2
#pragma unroll
                for (int s = 0; s < 2; ++s) {
                    const int j = lane + 32 * s;
                    S[oSnap + j] = (j < n) ? S[W.xc + j] * S[oL + j] : 0.0;
                }
                __syncwarp();
                const double SSE = echo_fit_sse(oSnap, O, n, lane, -1) + perp;
                if (SSE == 0.0) st |= MET2_ST_SSE_ZERO;
                // ---- starting set of the first Tikhonov solve
                Brent B;
                double lam = B.start(A.cfg.brent_lo, A.cfg.brent_hi, A.cfg.brent_xatol, A.cfg.maxfun);
                unsigned inP = 0u;
                double x[2] = {0.0, 0.0};
                bool block_drop = false;
                if (A.cfg.flags & MET2_T2_FLAG_FULL_START) {
                    // every column, feasible point xt_j = ct_j / (Gt_jj + lam) with ct = c / l, Gt_jj = G_jj / l_j^2
#pragma unroll
                    for (int s = 0; s < 2; ++s) {
                        const int j = lane + 32 * s;
                        if (j < n) {
                            const double il = S[oIL + j];
                            const double djj = fma(S[oG + j * ldg + j], il * il, lam);
                            x[s] = fmax(S[W.cc + j] * il / djj, 1e-300);
                            inP |= 1u << s;
                        }
                    }
                    for (int i = lane; i < tri(RD); i += 32) S[O.Mp + i] = S[oMf + i];
                    block_drop = true;
                } else {
                    // the plain solution's support and coefficients (scaled); M_P by rank-one terms
                    for (int i = lane; i < tri(RD); i += 32) S[O.Mp + i] = 0.0;
                    __syncwarp();
#pragma unroll
                    for (int s = 0; s < 2; ++s) {
                        const int j = lane + 32 * s;
                        const double xv = (j < n) ? S[oSnap + j] : 0.0;
                        if (xv > 0.0) {
                            x[s] = xv;
                            inP |= 1u << s;
                        }
                    }
                    for (int j = 0; j < n; ++j) {
                        const bool in = (__shfl_sync(FULL_MASK, inP, j & 31) >> (j >> 5)) & 1u;
                        if (in) echo_mp_rank1(O, j, 1.0, lane);
                    }
                }
                __syncwarp();
                // ---- Brent on |SSE(lam) - factor SSE| / SSE  (algorithms.py:219-233)
                double sse_snap = 0.0;
                int est = 0;
                while (true) {
                    echo_nnls<2>(W, O, n, lam, lane, inP, x, est, block_drop, true);
                    block_drop = false;
#pragma unroll
                    for (int s = 0; s < 2; ++s) S[W.xc + lane + 32 * s] = x[s];
                    __syncwarp();
                    // residual of the reduced system: bt - Ct xt = lam v exactly (push-through identity), v left in
                    // S[O.V..] by the solve echo_nnls accepted; the explicit product only after an itmax stop
                    double sse;
                    if (est & 1) {
                        sse = echo_fit_sse(W.xc, O, n, lane, -1) + perp;
                    } else {
                        const double ve = (lane < RD) ? S[O.V + lane] : 0.0;
                        sse = fma(lam * lam, warp_sum(ve * ve), perp);
                    }
                    const double cost = fabs(sse - A.cfg.factor * SSE) / SSE;
                    const double lam_eval = lam;
                    const bool more = B.feed(cost, lam);
                    if (B.xf == lam_eval) {
                        // the reference re-solves at Brent's best abscissa: keep that evaluation's solution instead
#pragma unroll
                        for (int s = 0; s < 2; ++s) S[oSnap + lane + 32 * s] = x[s];
                        sse_snap = sse;
                    }
                    __syncwarp();
                    if (!more) break;
                }
                lam = B.xf;
                // ---- hand out the best solution: fitted signal U (Ct xt), x = xt / l
                __syncwarp();
                (void)echo_fit_sse(oSnap, O, n, lane, O.V);
                __syncwarp();
                echo_expand<ME>(oU, O.V, m, lane, fit);
#pragma unroll
                for (int s = 0; s < 2; ++s) {
                    const int j = lane + 32 * s;
                    S[W.xc + j] = S[oSnap + j] * S[oIL + j];
                }
                __syncwarp();
                regv = (A.cfg.flags & MET2_T2_FLAG_REG_IS_LAMBDA) ? lam : sse_snap / SSE;
                if (nst || (est & 1)) st |= MET2_ST_ITMAX;
                if (est & 2) st |= MET2_ST_NOT_PD;
            }
            echo_outputs<2, ME>(A, v, W.xc, oLogT2, scomp, n, m, lane, st, km, regv, fit);
        }
    }
}

// ---------------------------------------------------------------------------------------------- fixed-lambda Tikhonov
// T2SPARC (algorithms.py:262-269 with reg = 1.8, motor...:138) in reduced echo space, nT2 <= 32 NC (the reference's 96
// bins: NC = 3).  One solve per voxel from the empty set: the factor of lam I is T = I / sqrt(lam), every entering /
// leaving column is one rank-one update of the RD x RD factor — no Gram matrix, no n x n factor (the Gram-domain
// kernel keeps tri(96) = 4 656 doubles per voxel and runs at three warps per SM).
// per-warp shared memory (doubles): Slots<2>(pmax RD) | M_P tri(RD) | raw signal (64) | bt (32) | v (32) | d (32) |
// x column space (32 NC)
template <int NC>
__host__ __device__ __forceinline__ int echo_tik_warp_doubles() {
    return (Slots<2>::doubles(RD) + tri(RD) + 64 + 32 + 32 + 32 + 32 * NC + 31) & ~31;
}
// CTA tables (doubles): Ct [32 NC][EC_LDD] | U [m][RD] | l | 1/l | logT2 (32 NC each) | comp
template <int NC>
__host__ __device__ __forceinline__ int echo_tik_table_doubles(int m) {
    return (32 * NC * EC_LDD + m * RD + 3 * 32 * NC + (32 * NC + 7) / 8 + EC_RC_DOUBLES + 31) & ~31;
}

template <int NC, int ME>
__global__ void __launch_bounds__(ECHO_TIK_MAX_THREADS, 1) t2_echo_tik_kernel(T2Args A) {
    __shared__ int s_tile, s_next, s_badL;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int n = A.cfg.nT2, m = A.cfg.nTE;
    constexpr int NCOL = 32 * NC;
    const int oCt = 0;
    const int oU = oCt + NCOL * EC_LDD;
    const int oL = oU + m * RD;
    const int oIL = oL + NCOL;
    const int oLogT2 = oIL + NCOL;
    unsigned char* scomp = reinterpret_cast<unsigned char*>(S + oLogT2 + NCOL);
    const int oRC = oLogT2 + NCOL + (NCOL + 7) / 8;
    const int wbase = echo_tik_table_doubles<NC>(m) + warp * echo_tik_warp_doubles<NC>();
    Slots<2> W;
    W.carve(wbase, RD);
    EchoOff O;
    O.Ct = oCt;
    O.RC = oRC;
    O.Mp = wbase + Slots<2>::doubles(RD);
    const int oM = O.Mp + tri(RD);
    O.B = oM + 64;
    O.V = O.B + 32;
    O.D = O.V + 32;
    const int oX = O.D + 32;
    const double lam = A.cfg.lambda_fixed;
    const double tdiag = 1.0 / sqrt(lam);

    if (threadIdx.x == 0) s_badL = 0;
    __syncthreads();
    echo_stage_diag(A, NCOL, n, oL, oIL, oLogT2, scomp, &s_badL);
    echo_stage_rc(oRC);
    const int ntiles = A.counters[0];

    while (true) {
        __syncthreads();
        if (threadIdx.x == 0) {
            s_tile = atomicAdd(&A.counters[1], 1);
            s_next = 0;
        }
        __syncthreads();
        const int tile = s_tile;
        if (tile >= ntiles) break;
        const bool badL = (s_badL != 0) || !(lam > 0.0);
        const int fa = A.tile_fa[tile];
        const int tstart = A.tile_start[tile], tcnt = A.tile_cnt[tile];
        const double* Cg = A.red_coef + (size_t)fa * n * RD;
        for (int i = threadIdx.x; i < NCOL * EC_LDD; i += blockDim.x) {
            const int j = i / EC_LDD, e = i - j * EC_LDD;
            S[oCt + i] = (j < n && e < RD) ? __ldg(Cg + j * RD + e) * S[oIL + j] : 0.0;
        }
        const double* Ug = A.red_basis + (size_t)fa * m * RD;
        for (int i = threadIdx.x; i < m * RD; i += blockDim.x) S[oU + i] = __ldg(Ug + i);
        __syncthreads();

        while (true) {
            int it = 0;
            if (lane == 0) it = atomicAdd(&s_next, 1);
            it = __shfl_sync(FULL_MASK, it, 0);
            if (it >= tcnt) break;
            const long long v = A.perm[tstart + it];
            unsigned st = load_signal<ME>(A.sig, v, m, oM, lane);
            const int fav = A.fa_index[v];
            const bool normalise = !(A.cfg.flags & MET2_T2_FLAG_NO_NORMALISE);
            const double km = normalise ? S[oM] : 1.0;
            if (!st && (!(km > 0.0) || fav < 0 || fav >= A.cfg.nA)) st = MET2_ST_SKIPPED;
            if (!st && badL) st = MET2_ST_SKIPPED | MET2_ST_ECHO_BAD_L;
            double fit[ME];
#pragma unroll
            for (int u = 0; u < ME; ++u) fit[u] = 0.0;
            if (!st) {
                __syncwarp();
#pragma unroll
                for (int u = 0; u < ME; ++u) {
                    const int e = lane + 32 * u;
                    if (e < m) S[oM + e] = S[oM + e] / km;
                }
                // empty set: M_P = 0, T = I / sqrt(lam)
                for (int i = lane; i < tri(RD); i += 32) {
                    S[O.Mp + i] = 0.0;
                    S[W.T + i] = 0.0;
                }
                __syncwarp();
                if (lane < RD) S[W.T + tri(lane) + lane] = tdiag;
                (void)echo_project<ME>(oU, oM, O.B, m, lane);
                __syncwarp();
                unsigned inP = 0u;
                double x[NC];
#pragma unroll
                for (int s = 0; s < NC; ++s) x[s] = 0.0;
                int est = 0;
                echo_nnls<NC>(W, O, n, lam, lane, inP, x, est, false, false);
#pragma unroll
                for (int s = 0; s < NC; ++s) S[oX + lane + 32 * s] = x[s];
                __syncwarp();
                (void)echo_fit_sse(oX, O, n, lane, O.V);
                __syncwarp();
                echo_expand<ME>(oU, O.V, m, lane, fit);
#pragma unroll
                for (int s = 0; s < NC; ++s) S[oX + lane + 32 * s] = x[s] * S[oIL + lane + 32 * s];
                __syncwarp();
                if (est & 1) st |= MET2_ST_ITMAX;
                if (est & 2) st |= MET2_ST_NOT_PD;
            }
            echo_outputs<NC, ME>(A, v, oX, oLogT2, scomp, n, m, lane, st, km, lam, fit);
        }
    }
}

template <int NC, int ME>
static int t2_launch_echo_tik(const T2Args& A, const Overrides& ov, cudaStream_t st) {
    const size_t tables = sizeof(double) * (size_t)echo_tik_table_doubles<NC>(A.cfg.nTE);
    const size_t per_warp = sizeof(double) * (size_t)echo_tik_warp_doubles<NC>();
    const int warps = echo_warps(tables, per_warp, ov, ECHO_TIK_MAX_THREADS);
    if (warps < 1) return set_error(MET2_ERR_UNSUPPORTED, "met2_t2_fit (echo space): tables do not fit in shared memory");
    const size_t smem = tables + per_warp * warps;
    int sms = sm_count();
    if (sms <= 0) sms = 148;
    cudaError_t e = cudaFuncSetAttribute(t2_echo_tik_kernel<NC, ME>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return set_error(MET2_ERR_CUDA, "t2_echo_tik attr (%zu B): %s", smem, cudaGetErrorString(e));
    MET2_LAUNCH(sms, warps * 32, smem, st, t2_echo_tik_kernel<NC, ME>)(A);
    count_launch();
    return check_launch("t2_echo_tik_kernel");
}

template <int ME>
static int t2_launch_echo_me(const T2Args& A, const Overrides& ov, cudaStream_t st) {
    const int n = A.cfg.nT2;
    if (A.cfg.method == MET2_REG_T2SPARC) {
        const int nc = (n + 31) / 32;
        if (nc <= 1) return t2_launch_echo_tik<1, ME>(A, ov, st);
        if (nc == 2) return t2_launch_echo_tik<2, ME>(A, ov, st);
        if (nc == 3) return t2_launch_echo_tik<3, ME>(A, ov, st);
        return t2_launch_echo_tik<4, ME>(A, ov, st);
    }
    const size_t tables = sizeof(double) * (size_t)echo_table_doubles(n, A.cfg.nTE);
    const size_t per_warp = sizeof(double) * (size_t)echo_warp_doubles();
    const int warps = echo_warps(tables, per_warp, ov);
    if (warps < 1) return set_error(MET2_ERR_UNSUPPORTED, "met2_t2_fit (echo space): tables do not fit in shared memory");
    const size_t smem = tables + per_warp * warps;
    int sms = sm_count();
    if (sms <= 0) sms = 148;
    cudaError_t e = cudaFuncSetAttribute(t2_echo_x2_kernel<ME>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return set_error(MET2_ERR_CUDA, "t2_echo attr (%zu B): %s", smem, cudaGetErrorString(e));
    MET2_LAUNCH(sms, warps * 32, smem, st, t2_echo_x2_kernel<ME>)(A);
    count_launch();
    return check_launch("t2_echo_x2_kernel");
}

}  // namespace MET2_ECHO_NS

int MET2_ECHO_LAUNCH(const T2Args& A, const Overrides& ov, cudaStream_t st) {
    if (A.cfg.nTE <= 32) return MET2_ECHO_NS::t2_launch_echo_me<1>(A, ov, st);
    return MET2_ECHO_NS::t2_launch_echo_me<2>(A, ov, st);
}

}  // namespace met2

#else   // MET2_ECHO_PART == 2

}  // namespace MET2_ECHO_NS
}  // namespace met2
#include "met2_t2_echo_reg_impl.cuh"

#endif
