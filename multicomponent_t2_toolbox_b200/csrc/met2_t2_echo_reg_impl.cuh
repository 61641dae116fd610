// met2_t2_echo_reg_impl.cuh — L-curve (algorithms.py:88-113) and BayesReg (bayesian_interpolation.py:84-126) in REDUCED
// ECHO SPACE for a diagonal regularisation matrix (I, InvT2).  Included by met2_t2_echo_impl.cuh (MET2_ECHO_PART == 2),
// inside its namespace: the Tikhonov NNLS solves are echo_nnls (rank-one updates of an RD x RD factor, RD = 16 / 24),
// the plain solve (lambda = 0: the first point of the L-curve grid, the noise estimate of BayesReg) is the Gram-domain
// nnls_gram in the same reduced space, as in t2_echo_x2_kernel.
//
// Why: the Gram-domain kernel keeps an n x n packed factor per voxel (tri(100) = 5 050 doubles at config 4's 100 bins) and
// BayesReg adds a dense n x n Cholesky factorisation per evidence evaluation, so config 4 ran at TWO warps per SM
// (profiles/r02_config4_ncu_summary.txt).  Here a voxel's state is ~6 KB (RD = 16, 60 bins) to ~12 KB (RD = 24, 100
// bins): 15-30 warps per SM.
//
// BayesReg evidence without the n x n factor.  With xt = l * f (l = diag L) and Ct = C diag(1/l) (RD x n):
//     A = beta B + beta x K = beta diag(l) (x I + Ct^T Ct) diag(l),   U = chol(A) = sqrt(beta) Ut diag(l),
//     Ut = upper Cholesky factor of At = x I + Ct^T Ct  (uniqueness of the factor with a positive diagonal), so
//     U f = sqrt(beta) Ut xt,   U_kk = sqrt(beta) l_k Ut_kk.
// At is diagonal plus rank RD, and its Cholesky factor has generator form: eliminating columns 0..j-1 leaves the Schur
// complement x I + Ct^T S_j Ct with an RD x RD state S_j (S_0 = I):
//     s = S_j ct_j,  a_j = x + ct_j . s  (= Ut_jj^2),  Ut_ji = (ct_i . s) / sqrt(a_j)  (i > j),  S_{j+1} = S_j - s s^T / a_j
// hence (Ut xt)_j = sqrt(a_j) xt_j + (s . sum_{i > j} xt_i ct_i) / sqrt(a_j): one forward sweep over the n columns with
// S_j in registers (RD^2 / 32 entries per lane), 2 RD^2 FMA per column instead of the (n - j)^2 / 2 of the dense
// factorisation, no n x n storage.  a_j >= x > 0: every pivot is a sum of positive terms up to the rounding of S_j
// (entries <= 1, absolute error ~1e-16 — the error class of the dense factorisation's late pivots).
//
// L-curve: the small end of the lambda grid stays in the Gram domain.  The triangle method (algorithms.py:150-206) looks
// at the angle between NEIGHBOURING grid points, which at lambda ~ 1e-8 differ by ~1e-8 relative: the echo-space solve
// of (lam I + M_P) with a rank-deficient M_P (condition number up to 4e14 for InvT2 at lam = 1e-8) is accurate to
// 1e-8 .. 2e-6 there, with errors that are independent from one grid point to the next, and produced a spurious corner
// at lambda <= 2.4e-8 in 531 of 552 960 voxels (InvT2; 1 with I) where the Gram-domain kernel agreed with the reference
// in all 121 voxels examined (profiles/r02_lcurve_arbiter.json).  Grid points below T2Args::lcurve_switch = 1e-5 are
// therefore solved by nnls_gram on G + lam K in the same reduced space (warm-started, supports of 4-10 columns), the
// rest in echo space.  The noise-to-difference ratio falls as 1 / lambda^2: at 1e-5 it is 6e-6 of its value at the
// largest failing lambda.  Measured over the whole config-2 volume with I and with InvT2 (2 x 552 960 voxels): the chosen
// corner equals the Gram-domain kernel's in every voxel for a switch at 1e-6, 1e-5, 1e-4 and 1e-3
// (profiles/r02_ab_lcurve_switch.json; T2 stage 348 / 394 / 413 / 441 ms with I against 290 ms all-echo and 565 ms
// Gram-domain).
#pragma once

namespace met2 {
namespace MET2_ECHO_NS {

constexpr int EV_RR = RD / 8;   // rows of the evidence state S_j per lane: rg + 8 a, rg = lane & 7
constexpr int EV_CC = RD / 4;   // columns per lane: cb EV_CC + b, cb = lane >> 3

constexpr int EV_LCURVE_PMAX = 32;          // positions of the Gram-domain factor of the L-curve kernel (one slot per lane)
template <int METHOD>
struct EchoRegPmax {
    static constexpr int value = (METHOD == MET2_REG_LCURVE) ? EV_LCURVE_PMAX : RD;
};

// per-warp shared memory (doubles): Slots<NC>(pmax) | M_P packed tri(RD) | raw signal, later the snapshot of the best /
// plain xt (max(64, 32 NC)) | bt, v, d (RD each) | L-curve: the two curves (MET2_MAX_LAMBDAS each)
template <int METHOD, int NC>
__host__ __device__ __forceinline__ int echo_reg_warp_doubles() {
    return (Slots<NC>::doubles(EchoRegPmax<METHOD>::value) + tri(RD) + (32 * NC > 64 ? 32 * NC : 64) + 3 * RD +
            (METHOD == MET2_REG_LCURVE ? 2 * MET2_MAX_LAMBDAS : 0) + 7) & ~7;
}
// CTA tables (doubles): G [n][ldg] (only when staged: NC == 2) | Ct [32 NC][EC_LDD] | U [m][RD] | l | 1/l | logT2 (32 NC
// each) | comp bytes | (row, column) bytes of the packed triangle | lambda grid (MET2_MAX_LAMBDAS) | K bands [5][32 NC]
template <int NC>
__host__ __device__ __forceinline__ int echo_reg_table_doubles(int n, int m) {
    return ((NC == 2 ? n * t2_ldg(n) : 0) + 32 * NC * EC_LDD + m * RD + 3 * 32 * NC + (32 * NC + 7) / 8 + EC_RC_DOUBLES +
            MET2_MAX_LAMBDAS + 5 * 32 * NC + 31) & ~31;
}

// -log evidence of bayesian_interpolation.py:107-126 at lambda = x for the Tikhonov-NNLS solution xt = l * f in
// S[W.xc + 0..n) (column j at offset j).  Scratch: W.gs (a_j), W.rs (s . suffix), W.xs (U_kk), W.cc (exchange buffer),
// O.D (Ct xt) — all free between two echo-space solves.
template <int NC>
__device__ __forceinline__ double echo_bayes_cost(const Slots<NC>& W, const EchoOff& O, int oL, int n, int m, int lane,
                                                  double x, double beta, double sse, double nrm, double log_det_L,
                                                  unsigned& st) {
    const int rg = lane & 7, cb = lane >> 3;
    const int oA = W.gs, oQ = W.rs, oUk = W.xs, oTmp = W.cc, oX = W.xc;
    (void)echo_fit_sse(oX, O, n, lane, O.D);    // Ct xt -> S[O.D ..]: the suffix sums start from the full product
    __syncwarp();
    double Sm[EV_RR][EV_CC], suf[EV_RR];
#pragma unroll
    for (int a = 0; a < EV_RR; ++a) {
        suf[a] = S[O.D + rg + 8 * a];
#pragma unroll
        for (int b = 0; b < EV_CC; ++b) Sm[a][b] = (rg + 8 * a == cb * EV_CC + b) ? 1.0 : 0.0;
    }
#pragma unroll 1
    for (int j = 0; j < n; ++j) {
        const int cj = O.Ct + j * EC_LDD;
        double ctc[EV_CC], ctr[EV_RR], s[EV_RR];
#pragma unroll
        for (int b = 0; b < EV_CC; b += 2) {
            const double2 t = *reinterpret_cast<const double2*>(S + cj + cb * EV_CC + b);
            ctc[b] = t.x;
            ctc[b + 1] = t.y;
        }
#pragma unroll
        for (int a = 0; a < EV_RR; ++a) ctr[a] = S[cj + rg + 8 * a];
        const double xj = S[oX + j];
        // s = S_j ct_j: partial sums over this lane's columns, then over the four column blocks
#pragma unroll
        for (int a = 0; a < EV_RR; ++a) {
            double acc = 0.0;
#pragma unroll
            for (int b = 0; b < EV_CC; ++b) acc = fma(Sm[a][b], ctc[b], acc);
            s[a] = acc;
        }
#pragma unroll
        for (int a = 0; a < EV_RR; ++a) {
            s[a] += __shfl_xor_sync(FULL_MASK, s[a], 8);
            s[a] += __shfl_xor_sync(FULL_MASK, s[a], 16);
        }
        // suffix sum_{i > j} xt_i ct_i, then the two dot products over the rows
        double q1 = 0.0, q2 = 0.0;
#pragma unroll
        for (int a = 0; a < EV_RR; ++a) {
            suf[a] = fma(-xj, ctr[a], suf[a]);
            q1 = fma(ctr[a], s[a], q1);
            q2 = fma(s[a], suf[a], q2);
        }
#pragma unroll
        for (int o = 1; o < 8; o <<= 1) {
            q1 += __shfl_xor_sync(FULL_MASK, q1, o);
            q2 += __shfl_xor_sync(FULL_MASK, q2, o);
        }
        const double aj = x + q1;
        // s in column layout through a double-buffered exchange (one barrier per column)
        const int ob = oTmp + (j & 1) * RD;
        if (cb == 0) {
#pragma unroll
            for (int a = 0; a < EV_RR; ++a) S[ob + rg + 8 * a] = s[a];
        }
        if (lane == 0) {
            S[oA + j] = aj;
            S[oQ + j] = q2;
        }
        __syncwarp();
        const double r = rcp_fast(aj);
#pragma unroll
        for (int b = 0; b < EV_CC; b += 2) {
            const double2 t = *reinterpret_cast<const double2*>(S + ob + cb * EV_CC + b);
            ctc[b] = t.x;
            ctc[b + 1] = t.y;
        }
#pragma unroll
        for (int a = 0; a < EV_RR; ++a) {
            const double sr = s[a] * r;
#pragma unroll
            for (int b = 0; b < EV_CC; ++b) Sm[a][b] = fma(-sr, ctc[b], Sm[a][b]);
        }
    }
    __syncwarp();
    // U f and diag U per column, lane = column
    const double sb = sqrt(beta);
    double series = 0.0;
    bool pd = true;
#pragma unroll
    for (int t = 0; t < NC; ++t) {
        const int j = lane + 32 * t;
        if (j < n) {
            const double aj = S[oA + j];
            if (!(aj > 0.0)) pd = false;
            const double ljj = sqrt(aj);
            const double uf = sb * fma(ljj, S[oX + j], S[oQ + j] / ljj);
            series += log(1.0 + erf(0.7071067811865475 * uf));
            S[oUk + j] = sb * ljj * S[oL + j];
        }
    }
    series = warp_sum(series);
    pd = __all_sync(FULL_MASK, pd);
    __syncwarp();
    if (!pd) st |= MET2_ST_NOT_PD;
    // det_U = prod(diag(U)) in np.prod's order (under- and overflow like the reference's)
    double det_u = 1.0;
    for (int k = 0; k < n; ++k) det_u *= S[oUk + k];
    const double ED = 0.5 * sse, EW = 0.5 * nrm;
    const double PI = 3.141592653589793;
    const double hn = n / 2.0, hm = m / 2.0;
    const double cost1 = beta * ED + beta * x * EW + log(det_u) - hn * log(PI / 2.0) - series;
    const double cost2 = hm * log(2.0 * PI) - hm * log(beta) + hn * log(PI) - hn * log(2.0 * beta * x) - log_det_L;
    __syncwarp();
    return pd ? (cost1 + cost2) : INFINITY;
}

// launch bounds (profiles/r02_ab_echo_warps.json): the L-curve is best at 640 threads (96 registers), BayesReg at 60 bins
// at 1024 (64 registers; 30 warps fit beside the tables); 100 bins: shared memory allows 12-15 warps -> 512 (128 registers)
template <int METHOD, int NC>
struct EchoRegThreads {
    static constexpr int value = (NC > 2) ? 512 : (METHOD == MET2_REG_BAYESREG ? 1024 : ECHO_MAX_THREADS);
};

template <int METHOD, int NC, int ME>
__global__ void __launch_bounds__(EchoRegThreads<METHOD, NC>::value, 1) t2_echo_reg_kernel(T2Args A) {
    static_assert(NC == 2 || NC == 4, "column slots");
    static_assert(METHOD == MET2_REG_LCURVE || METHOD == MET2_REG_BAYESREG, "method");
    constexpr bool GSH = (NC == 2);
    constexpr int NCOL = 32 * NC;
    constexpr int NSNAP = (NCOL > 64) ? NCOL : 64;
    __shared__ int s_tile, s_next, s_badL;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int n = A.cfg.nT2, m = A.cfg.nTE;
    const int ldg = GSH ? t2_ldg(n) : n;
    const int oG = 0;
    const int oCt = oG + (GSH ? n * ldg : 0);
    const int oU = oCt + NCOL * EC_LDD;
    const int oL = oU + m * RD;
    const int oIL = oL + NCOL;
    const int oLogT2 = oIL + NCOL;
    unsigned char* scomp = reinterpret_cast<unsigned char*>(S + oLogT2 + NCOL);
    const int oRC = oLogT2 + NCOL + (NCOL + 7) / 8;
    constexpr int PMAX = EchoRegPmax<METHOD>::value;
    const int oLam = oRC + EC_RC_DOUBLES;
    const int oKb = oLam + MET2_MAX_LAMBDAS;     // K = L^T L in 5-band form [5][n] (nnls_gram with reg)
    const int wbase = echo_reg_table_doubles<NC>(n, m) + warp * echo_reg_warp_doubles<METHOD, NC>();
    Slots<NC> W;
    W.carve(wbase, PMAX);
    EchoOff O;
    O.Ct = oCt;
    O.RC = oRC;
    O.Mp = wbase + Slots<NC>::doubles(PMAX);
    const int oM = O.Mp + tri(RD);
    O.B = oM + NSNAP;
    O.V = O.B + RD;
    O.D = O.V + RD;
    const int oSnap = oM;     // the raw signal is not needed once it is projected (bt) and km is in a register
    const int oLx = O.D + RD, oLy = oLx + MET2_MAX_LAMBDAS;   // L-curve: log residual / log norm per grid point

    if (threadIdx.x == 0) s_badL = 0;
    __syncthreads();
    echo_stage_diag(A, NCOL, n, oL, oIL, oLogT2, scomp, &s_badL);
    echo_stage_rc(oRC);
    if (METHOD == MET2_REG_LCURVE) {
        for (int i = threadIdx.x; i < A.cfg.nLambda; i += blockDim.x) S[oLam + i] = A.lambdas[i];
        for (int i = threadIdx.x; i < 5 * n; i += blockDim.x) S[oKb + i] = A.kband[i];
    }
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
        const double* Gg = A.G + (size_t)fa * n * n;
        if (GSH) {
            for (int i = threadIdx.x; i < n * n; i += blockDim.x) {
                const int r = i / n;
                S[oG + r * ldg + (i - r * n)] = __ldg(Gg + i);
            }
        }
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
                // ---- plain NNLS in the Gram domain (algorithms.py:55-82): c = D^T b = l * (Ct^T bt)
                {
                    double g[NC];
                    echo_gprod<NC>(O, O.B, lane, g);
#pragma unroll
                    for (int s = 0; s < NC; ++s) {
                        const int j = lane + 32 * s;
                        if (j < n) S[W.cc + j] = g[s] * S[oL + j];
                    }
                    __syncwarp();
                }
                set_dspace<NC>(W, Cg, O.B, lane);     // candidate test in the reduced space: rows of C, right-hand side bt
                // ---- lambda-search driver: a small state machine around ONE inlined Gram-domain call site (nnls_gram) and
                //      ONE inlined echo-space call site (echo_refactor + echo_nnls) — the kernel with a call site per use was
                //      18.8 k SASS instructions and instruction-fetch bound (config-2 L-curve 541 ms against 270 ms for the
                //      same counted work, DESIGN.md §6)
                //   PH_PLAIN : plain NNLS (algorithms.py:55-82) -> SSE0, support; BayesReg: beta
                //   PH_GRID  : L-curve grid (algorithms.py:88-113), below A.lcurve_switch in the Gram domain
                //   PH_FINAL : L-curve solve at the corner (algorithms.py:262-269)
                //   PH_BRENT : BayesReg evidence search (bayesian_interpolation.py:84-105)
                enum { PH_PLAIN = 0, PH_GRID = 1, PH_FINAL = 2, PH_BRENT = 3 };
                int phase = PH_PLAIN;
                int nst = 0, est = 0, p = 0, gi = 0;
                unsigned inP = 0u;
                double x[NC];
#pragma unroll
                for (int s = 0; s < NC; ++s) x[s] = 0.0;
                bool in_echo = false;
                double SSE0 = 0.0, beta = 0.0, lam_cur = 0.0, lam = 0.0;
                const int nl = A.cfg.nLambda;
                Brent B;
                while (true) {
                    double sse = SSE0, nrm = 0.0;
                    bool done = false;
                    if (METHOD == MET2_REG_LCURVE && phase != PH_PLAIN && !(lam_cur > 0.0)) {
                        // lambda_reg[0] = 0 (motor...:248-251): the plain solution, kept in the snapshot
                        double a = 0.0;
#pragma unroll
                        for (int s = 0; s < NC; ++s) {
                            const double xv = S[oSnap + lane + 32 * s];
                            a = fma(xv, xv, a);
                        }
                        nrm = warp_sum(a);
                        done = true;
                    } else if (phase == PH_PLAIN ||
                               (METHOD == MET2_REG_LCURVE && !in_echo && lam_cur < A.lcurve_switch && p < PMAX)) {
                        // Gram domain: the plain solve from the empty set (<= RD positions), or a Tikhonov solve on
                        // G + lam K from the carried-over positions (<= PMAX; a full factor sends the point to echo space).
                        // Cold-starting those points as well measured much slower (L-curve 293 -> 466 ms).
                        const bool plain = (METHOD == MET2_REG_BAYESREG) ? true : (phase == PH_PLAIN);   // BayesReg: compile-time
                        const int pn = nnls_gram<NC, GSH, 1>(W, oG, Gg, ldg, oKb, !plain, lam_cur, n, plain ? RD : PMAX, lane,
                                                              nst, plain ? 0 : p, false);
                        double a = 0.0;
#pragma unroll
                        for (int s = 0; s < NC; ++s) {
                            const int j = lane + 32 * s;
                            const double xv = (j < n) ? S[W.xc + j] * S[oL + j] : 0.0;     // xt = l * x
                            x[s] = (xv > 0.0) ? xv : 0.0;
                            a = fma(x[s], x[s], a);
                        }
                        __syncwarp();
#pragma unroll
                        for (int s = 0; s < NC; ++s) S[W.xc + lane + 32 * s] = x[s];
                        __syncwarp();
                        p = pn;
                        if (plain || pn < PMAX) {
                            nrm = warp_sum(a);
                            sse = echo_fit_sse(W.xc, O, n, lane, -1) + perp;     // |Ct xt - bt|^2 + |b_perp|^2
                            done = true;
                        }
                    }
                    if (!done) {
                        if (!in_echo) {
                            // enter echo space from the scaled solution xt in S[W.xc ..]: support, coefficients, M_P
                            inP = 0u;
#pragma unroll
                            for (int s = 0; s < NC; ++s) {
                                const double xv = S[W.xc + lane + 32 * s];
                                x[s] = (xv > 0.0) ? xv : 0.0;
                                if (xv > 0.0) inP |= 1u << s;
                            }
                            for (int i = lane; i < tri(RD); i += 32) S[O.Mp + i] = 0.0;
                            __syncwarp();
                            for (int j = 0; j < n; ++j) {
                                const bool in = (__shfl_sync(FULL_MASK, inP, j & 31) >> (j >> 5)) & 1u;
                                if (in) echo_mp_rank1(O, j, 1.0, lane);
                            }
                            __syncwarp();
                            in_echo = true;
                        }
                        echo_nnls<NC>(W, O, n, lam_cur, lane, inP, x, est, false, true);
                        double a = 0.0;
#pragma unroll
                        for (int s = 0; s < NC; ++s) {
                            S[W.xc + lane + 32 * s] = x[s];
                            a = fma(x[s], x[s], a);
                        }
                        __syncwarp();
                        nrm = warp_sum(a);       // |L f|^2 = |xt|^2
                        // bt - Ct xt = lam v exactly (push-through identity); the explicit product only after an itmax stop
                        if (est & 1) {
                            sse = echo_fit_sse(W.xc, O, n, lane, -1) + perp;
                        } else {
                            const double ve = (lane < RD) ? S[O.V + lane] : 0.0;
                            sse = fma(lam_cur * lam_cur, warp_sum(ve * ve), perp);
                        }
                    }
                    // ---- consume the solve
                    if (phase == PH_PLAIN) {
                        SSE0 = sse;
#pragma unroll
                        for (int s = 0; s < NC; ++s) S[oSnap + lane + 32 * s] = x[s];
                        __syncwarp();
                        if (METHOD == MET2_REG_BAYESREG) {
                            // bayesian_interpolation.py:84-105: beta from the plain solution, Brent over [1e-8, 2]
                            int nnz = 0;
#pragma unroll
                            for (int s = 0; s < NC; ++s)
                                if (x[s] > 0.0) ++nnz;
                            nnz = (int)__reduce_add_sync(FULL_MASK, (unsigned)nnz);
                            const double dof = fmax((double)(m - nnz), 1.0);
                            const double sigma = sqrt(SSE0 / dof);
                            beta = 1.0 / (sigma * sigma);
                            lam_cur = B.start(A.cfg.brent_lo, A.cfg.brent_hi, A.cfg.brent_xatol, A.cfg.maxfun);
                            phase = PH_BRENT;
                        } else {
                            gi = 0;
                            lam_cur = S[oLam];
                            phase = PH_GRID;
                        }
                    } else if (phase == PH_BRENT) {
                        const double cost = echo_bayes_cost<NC>(W, O, oL, n, m, lane, lam_cur, beta, sse, nrm, A.cfg.log_det_L, st);
                        const double lam_eval = lam_cur;
                        const bool more = B.feed(cost, lam_cur);
                        if (B.xf == lam_eval) {
                            // the reference re-solves at Brent's best abscissa: keep that evaluation's solution instead
#pragma unroll
                            for (int s = 0; s < NC; ++s) S[oSnap + lane + 32 * s] = x[s];
                        }
                        __syncwarp();
                        if (!more) {
                            lam = B.xf;
                            break;
                        }
                    } else if (phase == PH_GRID) {
                        if (lane == 0) {
                            S[oLx + gi] = log(sse + 1e-200);
                            S[oLy + gi] = log(nrm + 1e-200);
                        }
                        __syncwarp();
                        ++gi;
                        if (gi < nl) {
                            lam_cur = S[oLam + gi];
                        } else {
                            lam = S[oLam + select_corner_warp(oLx, oLy, nl, lane)];
                            if (!(lam > 0.0)) break;       // the plain solution, already in the snapshot
                            lam_cur = lam;
                            phase = PH_FINAL;
                        }
                    } else {   // PH_FINAL
#pragma unroll
                        for (int s = 0; s < NC; ++s) S[oSnap + lane + 32 * s] = x[s];
                        __syncwarp();
                        break;
                    }
                }
                // ---- hand out the solution in the snapshot: fitted signal U (Ct xt), x = xt / l
                __syncwarp();
                (void)echo_fit_sse(oSnap, O, n, lane, O.V);
                __syncwarp();
                echo_expand<ME>(oU, O.V, m, lane, fit);
#pragma unroll
                for (int s = 0; s < NC; ++s) {
                    const int j = lane + 32 * s;
                    S[W.xc + j] = S[oSnap + j] * S[oIL + j];
                }
                __syncwarp();
                regv = lam;
                if (nst || (est & 1)) st |= MET2_ST_ITMAX;
                if (est & 2) st |= MET2_ST_NOT_PD;
            }
            echo_outputs<NC, ME>(A, v, W.xc, oLogT2, scomp, n, m, lane, st, km, regv, fit);
        }
    }
}

template <int METHOD, int NC, int ME>
static int t2_launch_echo_reg_one(const T2Args& A, const Overrides& ov, cudaStream_t st) {
    const size_t tables = sizeof(double) * (size_t)echo_reg_table_doubles<NC>(A.cfg.nT2, A.cfg.nTE);
    const size_t per_warp = sizeof(double) * (size_t)echo_reg_warp_doubles<METHOD, NC>();
    const int warps = echo_warps(tables, per_warp, ov, EchoRegThreads<METHOD, NC>::value);
    if (warps < 1) return set_error(MET2_ERR_UNSUPPORTED, "met2_t2_fit (echo space): tables do not fit in shared memory");
    const size_t smem = tables + per_warp * warps;
    int sms = sm_count();
    if (sms <= 0) sms = 148;
    cudaError_t e = cudaFuncSetAttribute(t2_echo_reg_kernel<METHOD, NC, ME>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return set_error(MET2_ERR_CUDA, "t2_echo_reg attr (%zu B): %s", smem, cudaGetErrorString(e));
    MET2_LAUNCH(sms, warps * 32, smem, st, t2_echo_reg_kernel<METHOD, NC, ME>)(A);
    count_launch();
    return check_launch("t2_echo_reg_kernel");
}

template <int METHOD>
static int t2_launch_echo_reg_method(const T2Args& A, const Overrides& ov, cudaStream_t st) {
    const bool wide = A.cfg.nT2 > 64, me2 = A.cfg.nTE > 32;
    if (!wide && !me2) return t2_launch_echo_reg_one<METHOD, 2, 1>(A, ov, st);
    if (!wide && me2) return t2_launch_echo_reg_one<METHOD, 2, 2>(A, ov, st);
    if (wide && !me2) return t2_launch_echo_reg_one<METHOD, 4, 1>(A, ov, st);
    return t2_launch_echo_reg_one<METHOD, 4, 2>(A, ov, st);
}

}  // namespace MET2_ECHO_NS

int MET2_ECHO_LAUNCH(const T2Args& A, const Overrides& ov, cudaStream_t st) {
    if (A.cfg.method == MET2_REG_LCURVE) return MET2_ECHO_NS::t2_launch_echo_reg_method<MET2_REG_LCURVE>(A, ov, st);
    return MET2_ECHO_NS::t2_launch_echo_reg_method<MET2_REG_BAYESREG>(A, ov, st);
}

}  // namespace met2
