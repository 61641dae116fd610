// met2_fa.cu — flip-angle estimation for a batch of voxels (Step 2 of the reference orchestrator).
//
// Takes over flip_angle_algorithms/fa_estimation.py: compute_optimal_FA (:74-90, brute force),
// fitting_slice_FA_spline_method (:35-70) and the joblib loop that drives them (motor/motor_recon_met2_real_data.py:349-373).
//   kernel 1 (fa_search_kernel): residual norm of the plain NNLS fit for every search angle and voxel.  Angles are the
//       OUTER loop of each CTA: the ~59 KB of tables of one angle (D, D^T, G) are staged in shared memory once per
//       angle and CTA (the version that read them through L1/L2 spent its time on L2 latency), and every voxel's fit
//       is warm-started from its fit at the previous angle.
//   kernel 2 (fa_select_kernel): brute force -> the running arg-min of kernel 1; spline -> not-a-knot cubic through the
//       15 knot residuals, SciPy's bounded Brent on it, snap to the fine grid; then the NNLS at the chosen angle for
//       km = sum(f) and the per-warp partial sums of f (mean_T2_dist).
//   kernel 3: fixed-order reduction of those partial sums (deterministic for a given launch geometry).
#include <cmath>
#include <cstdio>
#include <cstdlib>

#include "met2_device.cuh"
#include "met2_host.h"

namespace met2 {

struct FaArgs {
    const double* sig;
    long long V;
    met2_fa_cfg cfg;
    const double *dic, *dicT, *G, *alphas;        // fine grid tables
    const double *dic_s, *dicT_s, *G_s, *knots;   // search tables (== fine for brute force)
    int nS;                                        // number of search angles
    int* fa_index;
    double *fa_deg, *km, *fsol_sum;
    unsigned* status;
    // workspace
    double* resid;      // spline: [V][nS]; brute force: best residual [V]
    double* wsp;        // [nK][nK] spline weights
    double* partial;    // [total warps][nT2]
    int* ws_p;          // [V] size of the positive set carried from the previous search angle (0 = none)
    int* ws_ix;         // [V][FA_CARRY] its columns
    double* ws_x;       // [V][FA_CARRY] its coefficients
    int pmax;
    // thread-per-voxel search (fa_search_thread_kernel): voxels it hands back to the warp-per-voxel kernel
    int* ovf_list;      // [V]
    int* ovf_count;     // [1] number of entries; the warp kernel reads it when vlist is set
    const int* vlist;   // warp kernel: nullptr = all V voxels, else the voxels ovf_list[0 .. *ovf_count)
    int thread_pcap;    // largest positive set the thread kernel keeps (<= FT_PM; tests lower it to force hand-backs)
};

constexpr int FA_CARRY = 16;   // supports of the plain fits have 3-8 columns; larger ones restart cold

constexpr int FA_WARPS = 8;

// per-warp shared memory in doubles: NNLS slots + signal ms[64]
template <int NS>
__host__ __device__ __forceinline__ int fa_warp_doubles(int pmax) {
    return (Slots<NS>::doubles(pmax) + 64 + 31) & ~31;
}

constexpr int FA_SEARCH_WARPS = 16;

__host__ __device__ __forceinline__ int fa_ldg(int n) { return (n + 1) & ~1; }
// staged tables of one angle, in doubles: D [m][n], Dt [n][m], G [n][ldg]
__host__ __device__ __forceinline__ int fa_table_doubles(int n, int m) { return (2 * m * n + n * fa_ldg(n) + 31) & ~31; }

template <int NS, int ME>
__global__ void __launch_bounds__(FA_SEARCH_WARPS * 32, 1) fa_search_kernel(FaArgs A) {
    // a plain solve has at most min(nT2, nTE) <= 32 ME positive columns: position-space loops of ME slots, not NS
    constexpr int FA_PS = (ME < NS) ? ME : NS;
    __shared__ int s_next;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int n = A.cfg.nT2, m = A.cfg.nTE;
    const int ldg = fa_ldg(n);
    const int oD = 0, oDt = m * n, oG = 2 * m * n;
    Slots<NS> W;
    const int wbase = fa_table_doubles(n, m) + warp * fa_warp_doubles<NS>(A.pmax);
    W.carve(wbase, A.pmax);
    const int oM = wbase + Slots<NS>::doubles(A.pmax);
    // list mode: only the voxels the thread-per-voxel kernel handed back (usually none: leave before staging anything)
    const long long Vn = A.vlist ? (long long)*A.ovf_count : A.V;
    const long long chunk = (Vn + gridDim.x - 1) / gridDim.x;
    const long long v0 = (long long)blockIdx.x * chunk;
    const long long v1 = (v0 + chunk < Vn) ? v0 + chunk : Vn;
    if (v0 >= v1) return;
    const bool brute = (A.cfg.method == MET2_FA_BRUTE_FORCE);
    for (int a = 0; a < A.nS; ++a) {
        {
            const double* D = A.dic_s + (size_t)a * m * n;
            const double* Dt = A.dicT_s + (size_t)a * n * m;
            const double* G = A.G_s + (size_t)a * n * n;
            for (int i = threadIdx.x; i < m * n; i += blockDim.x) {
                S[oD + i] = __ldg(D + i);
                S[oDt + i] = __ldg(Dt + i);
            }
            for (int i = threadIdx.x; i < n * n; i += blockDim.x) {
                const int r = i / n;
                S[oG + r * ldg + (i - r * n)] = __ldg(G + i);
            }
        }
        if (threadIdx.x == 0) s_next = 0;
        __syncthreads();
        // the warps pull the CTA's voxels one at a time (a static deal left them waiting for the slowest warp at the
        // barrier that ends every angle: 1.3 stalled warps per issue in profiles/r02_fa_*_ncu_summary.txt)
        while (true) {
            int iv = 0;
            if (lane == 0) iv = atomicAdd(&s_next, 1);
            iv = __shfl_sync(FULL_MASK, iv, 0);
            if (v0 + iv >= v1) break;
            const long long v = A.vlist ? (long long)A.vlist[v0 + iv] : v0 + iv;
            unsigned st = load_signal<ME>(A.sig, v, m, oM, lane);
            if (st) continue;
            compute_c_sh<NS>(W, oD, oM, m, n, lane);
            // warm start from the fit at the previous search angle (same voxel, neighbouring dictionary): the residual
            // norm of the NNLS optimum does not depend on the starting point
            int p0 = 0;
            if (a > 0) {
                p0 = A.ws_p[v];
                if (lane < p0) {
                    SI(W.ix, lane) = A.ws_ix[v * FA_CARRY + lane];
                    S[W.xs + lane] = A.ws_x[v * FA_CARRY + lane];
                }
                __syncwarp();
            }
            int nst = 0;
            set_dspace<NS>(W, A.dicT_s + (size_t)a * n * m, oM, lane);
            int p = nnls_gram<NS, true, FA_PS>(W, oG, nullptr, ldg, 0, false, 0.0, n, m, lane, nst, p0);
            if (a + 1 < A.nS) {
                const bool keep = (p <= FA_CARRY);
                if (keep && lane < p) {
                    A.ws_ix[v * FA_CARRY + lane] = SI(W.ix, lane);
                    A.ws_x[v * FA_CARRY + lane] = S[W.xs + lane];
                }
                if (lane == 0) A.ws_p[v] = keep ? p : 0;
            }
            double fit[ME];
            double sse = fit_and_sse_sh<NS, ME>(W, oDt, oM, m, p, lane, fit);
            double rnorm = sqrt(sse);
            if (lane == 0) {
                if (brute) {
                    // np.argmin: first minimum (fa_estimation.py:83)
                    if (a == 0 || rnorm < A.resid[v]) {
                        A.resid[v] = rnorm;
                        A.fa_index[v] = a;
                    }
                } else {
                    A.resid[v * A.nS + a] = rnorm;
                }
                if (nst) atomicOr(&A.status[v], MET2_ST_ITMAX);
            }
            __syncwarp();
        }
        __syncthreads();   // all warps are done with this angle's tables
    }
}

// ------------------------------------------------------------------------------------------------ thread per voxel
// The search solves plain NNLS problems whose optimal supports have 2-7 columns (measured on the config-2 phantom:
// 22 500 solves, none above 7): a warp per voxel leaves most lanes idle in every position-space step and spends its
// instructions on warp collectives and barriers (4 100 warp-instructions per warm-started solve, FP64 pipe 14 % busy,
// profiles/r02_config2_kernels_ncu_summary.txt).  Here ONE THREAD owns a voxel through all search angles:
//   * its signal b and the current residual r = b - D_P x live in registers (MR echoes, zero padded);
//   * the tables of one angle — D^T [n][MR + 2] and G [n][n] — are staged once per CTA and angle; the dual
//     w_j = d_j . r of ALL columns is a loop every thread runs in lock step, so each 128-bit shared-memory load is a
//     broadcast (one wavefront feeds 64 FMAs) and no per-voxel copy of c = D^T b or of w exists;
//   * the least-squares step on the positive set is taken in correction form, z = x + (G_PP)^-1 D_P^T r, with the
//     Cholesky factor of G_PP (at most PM x PM, packed, one column of shared memory per thread: conflict-free for any
//     index) — the right-hand side is a D-space residual, so the Gram-domain factor only has to be good enough for a
//     correction and the accuracy is that of iterative refinement;
//   * Lawson-Hanson's control flow is the one of nnls_gram (met2_nnls.cuh): first-maximum pivot, the two acceptance
//     tests of nnls.f (with the D-space evaluation of nearly dependent candidates), interpolation loop, itmax = 3 n,
//     warm start from the support and coefficients of the previous angle.
// A voxel whose positive set would exceed PM columns, that runs into itmax or meets a non-positive pivot is handed to
// the warp-per-voxel kernel (ovf_list), which redoes all its angles.
constexpr int FT_MAX_THREADS = 256;
constexpr int FT_PM = 8;

template <int MR>
__host__ __device__ __forceinline__ int ft_table_doubles(int n) {
    return (((n + 3) & ~3) * (MR + 2) + n * n + 1) & ~1;
}
// per thread, one contiguous block: L tri(PM) | x | z | g | dinv (PM each) | ix (PM ints); the stride is odd, so the 16
// threads of a half warp reading the same entry of their blocks hit 16 different 8-byte bank pairs
__host__ __device__ __forceinline__ int ft_thread_doubles() { return (tri(FT_PM) + 4 * FT_PM + FT_PM / 2) | 1; }

template <int MR>
__global__ void __launch_bounds__(FT_MAX_THREADS, 1) fa_search_thread_kernel(FaArgs A) {
    constexpr int PM = FT_PM;
    constexpr int LDD = MR + 2;     // even: 16-byte rows for the broadcast loads; 34 / 50 / 66 spread divergent rows over banks
    const int tid = threadIdx.x, T = blockDim.x;
    const int n = A.cfg.nT2, m = A.cfg.nTE;
    const int n4 = (n + 3) & ~3;
    const int oD = 0;
    const int oG = oD + n4 * LDD;
    const int oL = ft_table_doubles<MR>(n) + tid * ft_thread_doubles();
    const int oX = oL + tri(PM);
    const int oZ = oX + PM;
    const int oGv = oZ + PM;
    const int oDi = oGv + PM;
    const int oIx = oDi + PM;
    const bool brute = (A.cfg.method == MET2_FA_BRUTE_FORCE);
    const int itmax = 3 * n;
    const int mn = (m < n) ? m : n;
    const int pcap = (A.thread_pcap < mn) ? A.thread_pcap : mn;
#define FT_L(i, k) S[oL + tri(i) + (k)]
#define FT_X(i) S[oX + (i)]
#define FT_Z(i) S[oZ + (i)]
#define FT_GV(i) S[oGv + (i)]
#define FT_DI(i) S[oDi + (i)]
#define FT_IX(i) SI(oIx, (i))
    // The CTA owns a contiguous chunk of voxels.  Per angle its threads PULL voxels from a shared counter and advance them
    // in lock step, one Lawson-Hanson step per tick: a thread that finishes its voxel takes the next one at once, so the
    // warp stays full whatever the number of steps each voxel needs (first version: a thread kept its voxel through all
    // angles and every warp waited for its slowest voxel at each angle — 7.4 active threads per executed instruction).
    __shared__ int s_next;
    const long long chunk = (A.V + gridDim.x - 1) / gridDim.x;
    const long long v0 = (long long)blockIdx.x * chunk;
    const long long v1 = (v0 + chunk < A.V) ? v0 + chunk : A.V;
    const int cnt = (int)(v1 - v0);
    enum { NEED_W = 0, INNER = 1, TRIAL = 2 };
    for (int a = 0; a < A.nS; ++a) {
        __syncthreads();
        {
            const double* Dt = A.dicT_s + (size_t)a * n * m;
            const double* G = A.G_s + (size_t)a * n * n;
            for (int i = tid; i < n4 * LDD; i += T) {
                const int j = i / LDD, e = i - j * LDD;
                S[oD + i] = (j < n && e < m) ? __ldg(Dt + j * m + e) : 0.0;
            }
            for (int i = tid; i < n * n; i += T) S[oG + i] = __ldg(G + i);
            if (tid == 0) s_next = 0;
        }
        __syncthreads();
        bool active = false;
        long long v = 0;
        double b[MR], r[MR];
        int p = 0, nfact = 0, iter = 0, state = NEED_W;
        unsigned long long in0 = 0ull, in1 = 0ull, rej0 = 0ull, rej1 = 0ull;
        double sse = 0.0;
        // r = b - D_P x and its squared norm
        auto residual = [&]() {
#pragma unroll
            for (int e = 0; e < MR; ++e) r[e] = b[e];
            #pragma unroll 1
            for (int i = 0; i < p; ++i) {
                const double xi = FT_X(i);
                const int row = oD + FT_IX(i) * LDD;
#pragma unroll
                for (int e = 0; e < MR; e += 2) {
                    const double2 d = *reinterpret_cast<const double2*>(S + row + e);
                    r[e] = fma(-xi, d.x, r[e]);
                    r[e + 1] = fma(-xi, d.y, r[e + 1]);
                }
            }
            double s0 = 0.0, s1 = 0.0;
#pragma unroll
            for (int e = 0; e < MR; e += 2) {
                s0 = fma(r[e], r[e], s0);
                s1 = fma(r[e + 1], r[e + 1], s1);
            }
            sse = s0 + s1;
        };
        // Least-squares step on positions 0 .. pp-1 from the current r: g = D_P^T r, rows nfact .. pp-1 of the Cholesky
        // factor, z = x + (L L^T)^-1 g.  trial: position pp-1 is a candidate under the acceptance tests of nnls.f.
        // Returns 1 = fine, 0 = candidate rejected (nothing changed), -1 = not positive definite.  No early exits: the
        // threads of a warp walk through the same sequence of loops and only their trip counts differ.
        auto solve = [&](int pp, bool trial) -> int {
            #pragma unroll 1
            for (int i = 0; i < pp; ++i) {
                const int row = oD + FT_IX(i) * LDD;
                double g0 = 0.0, g1 = 0.0;
#pragma unroll
                for (int e = 0; e < MR; e += 2) {
                    const double2 d = *reinterpret_cast<const double2*>(S + row + e);
                    g0 = fma(d.x, r[e], g0);
                    g1 = fma(d.y, r[e + 1], g1);
                }
                FT_GV(i) = g0 + g1;
            }
            bool bad = false, rejected = false;
            double rho2c = 1.0, gjjc = 1.0, s1c = 0.0;
            #pragma unroll 1
            for (int i = nfact; i < pp; ++i) {
                const int ci = FT_IX(i);
                double s1 = 0.0;
                #pragma unroll 1
                for (int k = 0; k < i; ++k) {
                    double sacc = S[oG + ci * n + FT_IX(k)];
                    #pragma unroll 1
                    for (int q = 0; q < k; ++q) sacc = fma(-FT_L(i, q), FT_L(k, q), sacc);
                    const double lik = sacc * FT_DI(k);
                    FT_L(i, k) = lik;
                    s1 = fma(lik, lik, s1);
                }
                const double gjj = S[oG + ci * n + ci];
                double rho2 = gjj - s1;
                if (trial && i == pp - 1) {
                    rho2c = rho2;
                    gjjc = gjj;
                    s1c = s1;
                } else {
                    if (!(rho2 > 0.0)) {
                        bad = true;
                        rho2 = 1.0;
                    }
                    FT_DI(i) = rsqrt_fast(rho2);
                }
            }
            if (trial) {
                const int i = pp - 1;
                if (i > 0 && rho2c < 1e-12 * gjjc) {
                    // nearly dependent on the set: the Gram form cannot resolve rho^2 / G_jj below ~1e-16 while nnls.f
                    // accepts down to ~5e-27 (DESIGN.md §5) — a = L^-T l = (G_PP)^-1 G_Pj, rho^2 = |d_j - D_P a|^2 in
                    // D-space.  (Between 1e-12 and the warp kernel's 1e-10 the Gram value has three digits and the right
                    // sign; its error moves z along the nearly dependent direction only, where the residual does not
                    // change.)  The residual registers hold q: r is rebuilt from x before its next use.
                    #pragma unroll 1
                    for (int k = i - 1; k >= 0; --k) {
                        double acc = FT_L(i, k);
                        #pragma unroll 1
                        for (int q = k + 1; q < i; ++q) acc = fma(-FT_L(q, k), FT_Z(q), acc);
                        FT_Z(k) = acc * FT_DI(k);
                    }
                    {
                        const int row = oD + FT_IX(i) * LDD;
#pragma unroll
                        for (int e = 0; e < MR; e += 2) {
                            const double2 d = *reinterpret_cast<const double2*>(S + row + e);
                            r[e] = d.x;
                            r[e + 1] = d.y;
                        }
                    }
                    #pragma unroll 1
                    for (int k = 0; k < i; ++k) {
                        const double ak = FT_Z(k);
                        const int row = oD + FT_IX(k) * LDD;
#pragma unroll
                        for (int e = 0; e < MR; e += 2) {
                            const double2 d = *reinterpret_cast<const double2*>(S + row + e);
                            r[e] = fma(-ak, d.x, r[e]);
                            r[e + 1] = fma(-ak, d.y, r[e + 1]);
                        }
                    }
                    double q0 = 0.0, q1 = 0.0;
#pragma unroll
                    for (int e = 0; e < MR; e += 2) {
                        q0 = fma(r[e], r[e], q0);
                        q1 = fma(r[e + 1], r[e + 1], q1);
                    }
                    rho2c = q0 + q1;
                }
                if (!(rho2c > 0.0) || !(rho2c > 1.2e-28 * s1c)) {
                    rejected = true;
                    rho2c = 1.0;
                }
                FT_DI(i) = rsqrt_fast(rho2c);
            }
            // forward substitution y = L^-1 g (y in the z column)
            #pragma unroll 1
            for (int i = 0; i < pp; ++i) {
                double acc = FT_GV(i);
                #pragma unroll 1
                for (int k = 0; k < i; ++k) acc = fma(-FT_L(i, k), FT_Z(k), acc);
                FT_Z(i) = acc * FT_DI(i);
            }
            if (trial && !(FT_Z(pp - 1) > 0.0)) rejected = true;   // "ztest": the entering coefficient must be positive
            // backward substitution dz = L^-T y, z = x + dz
            #pragma unroll 1
            for (int i = pp - 1; i >= 0; --i) {
                double acc = FT_Z(i);
                #pragma unroll 1
                for (int k = i + 1; k < pp; ++k) acc = fma(-FT_L(k, i), FT_Z(k), acc);
                FT_Z(i) = acc * FT_DI(i);
            }
            #pragma unroll 1
            for (int i = 0; i < pp; ++i) FT_Z(i) += FT_X(i);
            if (bad) return -1;
            if (rejected) return 0;
            nfact = pp;
            return 1;
        };
        bool fin = false, ovf = false;
        // One pass of the interpolation loop on the solve just made: accept z (-> NEED_W) or step towards it and drop the
        // blocking position and every x_i <= 0 (-> INNER: solve again on the smaller set).
        auto after_solve = [&]() {
            ++iter;
            if (iter > itmax) {   // nnls.f stops with the current x; the warp kernel reproduces that and its status bit
                fin = ovf = true;
                return;
            }
            double alpha = 2.0;
            int jb = -1;
            #pragma unroll 1
            for (int i = 0; i < p; ++i) {
                const double zi = FT_Z(i);
                if (zi <= 0.0) {
                    const double xi = FT_X(i);
                    const double tt = xi / (xi - zi);
                    if (tt < alpha) {
                        alpha = tt;
                        jb = i;
                    }
                }
            }
            if (jb < 0) {
                #pragma unroll 1
                for (int i = 0; i < p; ++i) FT_X(i) = FT_Z(i);
                state = NEED_W;
            } else {
                int q = 0;
                int firstout = p;
                #pragma unroll 1
                for (int i = 0; i < p; ++i) {
                    const double xo = FT_X(i);
                    const double xi = xo + alpha * (FT_Z(i) - xo);
                    const int ci = FT_IX(i);
                    if (i == jb || xi <= 0.0) {
                        if (ci < 64) in0 &= ~(1ull << ci); else in1 &= ~(1ull << (ci - 64));
                        if (i < firstout) firstout = i;
                    } else {
                        FT_X(q) = xi;
                        FT_IX(q) = ci;
                        ++q;
                    }
                }
                p = q;
                if (firstout < nfact) nfact = firstout;
                state = INNER;
            }
        };
        while (true) {
            // ---- refill: an idle thread takes the next voxel of the chunk
            while (!active) {
                const int idx = atomicAdd(&s_next, 1);
                if (idx >= cnt) break;
                v = v0 + idx;
                int p0 = 0;
                if (a > 0) {
                    p0 = A.ws_p[v];
                    if (p0 < 0) continue;   // not fitted (empty / non-finite signal) or handed to the warp kernel
                }
                double ssum = 0.0;
                bool bad = false;
#pragma unroll
                for (int e = 0; e < MR; ++e) {
                    b[e] = (e < m) ? A.sig[v * m + e] : 0.0;
                    ssum += b[e];
                    if (!isfinite(b[e])) bad = true;
                }
                if (bad || !(ssum > 0.0)) {   // fa_estimation.py:100; the select kernel writes this voxel's outputs
                    A.ws_p[v] = -1;
                    continue;
                }
                // warm start from the fit at the previous search angle (same voxel, neighbouring dictionary): the
                // residual norm of the NNLS optimum does not depend on the starting point
                p = p0;
                in0 = in1 = rej0 = rej1 = 0ull;
                #pragma unroll 1
                for (int i = 0; i < p; ++i) {
                    const int ci = A.ws_ix[v * FA_CARRY + i];
                    FT_IX(i) = ci;
                    FT_X(i) = A.ws_x[v * FA_CARRY + i];
                    if (ci < 64) in0 |= 1ull << ci; else in1 |= 1ull << (ci - 64);
                }
                nfact = 0;
                iter = 0;
                state = (p > 0) ? INNER : NEED_W;   // the interpolation loop runs first on a carried set (nnls_gram, p0 > 0)
                fin = ovf = false;
                active = true;
            }
            if (!__any_sync(FULL_MASK, active)) break;
            // ---- solve phase: the acceptance solve of a candidate (TRIAL) and the re-solves of the interpolation loop
            //      (INNER), until every voxel of the warp waits for a new candidate
            while (__any_sync(FULL_MASK, active && !fin && state != NEED_W)) {
                if (active && !fin && state != NEED_W) {
                    const bool trial = (state == TRIAL);
                    if (!trial) residual();   // TRIAL: x has not moved since the w pass
                    const int rc = solve(trial ? p + 1 : p, trial);
                    if (rc > 0) {
                        if (trial) {
                            const int bj = FT_IX(p);
                            if (bj < 64) in0 |= 1ull << bj; else in1 |= 1ull << (bj - 64);
                            ++p;
                            rej0 = rej1 = 0ull;
                        }
                        after_solve();
                    } else if (rc == 0 && trial) {
                        const int bj = FT_IX(p);
                        if (bj < 64) rej0 |= 1ull << bj; else rej1 |= 1ull << (bj - 64);   // the next best candidate
                        state = NEED_W;
                    } else {
                        fin = ovf = true;
                    }
                }
                __syncwarp();
            }
            // ---- w phase: dual of every column, entering candidate (first maximum over the zero set minus rejected ones)
            if (active && !fin) {
                residual();
                if (p >= n || p >= m) {
                    fin = true;
                } else {
                    double bv = 0.0;
                    int bj = -1;
                    for (int j0 = 0; j0 < n4; j0 += 4) {
                        double w0 = 0.0, w1 = 0.0, w2 = 0.0, w3 = 0.0, u0 = 0.0, u1 = 0.0, u2 = 0.0, u3 = 0.0;
                        const int row = oD + j0 * LDD;
#pragma unroll
                        for (int e = 0; e < MR; e += 2) {
                            const double2 d0 = *reinterpret_cast<const double2*>(S + row + e);
                            const double2 d1 = *reinterpret_cast<const double2*>(S + row + LDD + e);
                            const double2 d2 = *reinterpret_cast<const double2*>(S + row + 2 * LDD + e);
                            const double2 d3 = *reinterpret_cast<const double2*>(S + row + 3 * LDD + e);
                            w0 = fma(d0.x, r[e], w0); u0 = fma(d0.y, r[e + 1], u0);
                            w1 = fma(d1.x, r[e], w1); u1 = fma(d1.y, r[e + 1], u1);
                            w2 = fma(d2.x, r[e], w2); u2 = fma(d2.y, r[e + 1], u2);
                            w3 = fma(d3.x, r[e], w3); u3 = fma(d3.y, r[e + 1], u3);
                        }
                        w0 += u0; w1 += u1; w2 += u2; w3 += u3;
                        const unsigned ex = (unsigned)(((j0 < 64) ? ((in0 | rej0) >> j0) : ((in1 | rej1) >> (j0 - 64))) & 0xfull);
                        if (!(ex & 1u) && w0 > bv) { bv = w0; bj = j0; }
                        if (!(ex & 2u) && w1 > bv) { bv = w1; bj = j0 + 1; }
                        if (!(ex & 4u) && w2 > bv) { bv = w2; bj = j0 + 2; }
                        if (!(ex & 8u) && w3 > bv) { bv = w3; bj = j0 + 3; }
                    }
                    if (bj < 0) {
                        fin = true;
                    } else if (p >= pcap) {   // the set would outgrow this kernel's factor
                        fin = ovf = true;
                    } else {
                        FT_IX(p) = bj;
                        FT_X(p) = 0.0;
                        state = TRIAL;
                    }
                }
            }
            __syncwarp();
            // ---- results of the voxels that are done with this angle
            if (active && fin) {
                if (ovf) {
                    A.ws_p[v] = -1;
                    const int k = atomicAdd(A.ovf_count, 1);
                    A.ovf_list[k] = (int)v;
                } else {
                    const double rnorm = sqrt(sse);
                    if (brute) {
                        // np.argmin: first minimum (fa_estimation.py:83)
                        if (a == 0 || rnorm < A.resid[v]) {
                            A.resid[v] = rnorm;
                            A.fa_index[v] = a;
                        }
                    } else {
                        A.resid[v * A.nS + a] = rnorm;
                    }
                    if (a + 1 < A.nS) {
                        A.ws_p[v] = p;
                        #pragma unroll 1
                        for (int i = 0; i < p; ++i) {
                            A.ws_ix[v * FA_CARRY + i] = FT_IX(i);
                            A.ws_x[v * FA_CARRY + i] = FT_X(i);
                        }
                    }
                }
                active = false;
            }
        }
    }
#undef FT_L
#undef FT_X
#undef FT_Z
#undef FT_GV
#undef FT_DI
#undef FT_IX
}

// Not-a-knot cubic spline as a linear map from knot values to knot second derivatives: Msec = Wsp * y.
// (scipy.interpolate.interp1d(kind='cubic') -> make_interp_spline(k=3), default not-a-knot; fa_estimation.py:54.)
// Gauss-Jordan with partial pivoting on the augmented K x 2K system, one warp: lane j owns columns j and j + 32 of every
// row, so each entry sees exactly the operations (and the order) of a serial elimination.  (Round 1 ran it on ONE
// thread with the matrix in a 16.6 KB local-memory frame: 112 us in front of every FA call.)
__global__ void __launch_bounds__(32, 1) spline_weights_kernel(const double* __restrict__ knots, int K,
                                                               double* __restrict__ wsp) {
    constexpr int LD = 2 * MET2_MAX_KNOTS + 1;
    __shared__ double Aug[MET2_MAX_KNOTS * LD];
    __shared__ double h[MET2_MAX_KNOTS];
    const int lane = threadIdx.x;
    const int W2 = 2 * K;
    for (int i = 0; i < K; ++i)
        for (int j = lane; j < W2; j += 32) Aug[i * LD + j] = 0.0;
    if (lane + 1 < K) h[lane] = knots[lane + 1] - knots[lane];
    __syncwarp();
    if (lane == 0) {
        Aug[0] = -1.0 / h[0];
        Aug[1] = 1.0 / h[0] + 1.0 / h[1];
        Aug[2] = -1.0 / h[1];
        Aug[(K - 1) * LD + K - 3] = -1.0 / h[K - 3];
        Aug[(K - 1) * LD + K - 2] = 1.0 / h[K - 3] + 1.0 / h[K - 2];
        Aug[(K - 1) * LD + K - 1] = -1.0 / h[K - 2];
    }
    if (lane >= 1 && lane + 1 < K) {
        const int i = lane;
        Aug[i * LD + i - 1] = h[i - 1] / 6.0;
        Aug[i * LD + i] = (h[i - 1] + h[i]) / 3.0;
        Aug[i * LD + i + 1] = h[i] / 6.0;
        Aug[i * LD + K + i - 1] = 1.0 / h[i - 1];
        Aug[i * LD + K + i] = -1.0 / h[i - 1] - 1.0 / h[i];
        Aug[i * LD + K + i + 1] = 1.0 / h[i];
    }
    __syncwarp();
    for (int c = 0; c < K; ++c) {
        int piv = c;
        double best = fabs(Aug[c * LD + c]);
        for (int r = c + 1; r < K; ++r)
            if (fabs(Aug[r * LD + c]) > best) {
                best = fabs(Aug[r * LD + c]);
                piv = r;
            }
        __syncwarp();
        if (piv != c) {
            for (int j = lane; j < W2; j += 32) {
                double t = Aug[c * LD + j];
                Aug[c * LD + j] = Aug[piv * LD + j];
                Aug[piv * LD + j] = t;
            }
            __syncwarp();
        }
        const double inv = 1.0 / Aug[c * LD + c];
        __syncwarp();
        for (int j = lane; j < W2; j += 32) Aug[c * LD + j] *= inv;
        __syncwarp();
        const double f_own = (lane < K) ? Aug[lane * LD + c] : 0.0;   // column c of every row, before it is eliminated
        __syncwarp();
        for (int r = 0; r < K; ++r) {
            const double f = __shfl_sync(0xffffffffu, f_own, r);
            if (r == c || f == 0.0) continue;
            for (int j = lane; j < W2; j += 32) Aug[r * LD + j] -= f * Aug[c * LD + j];
        }
        __syncwarp();
    }
    for (int i = 0; i < K; ++i)
        for (int j = lane; j < K; j += 32) wsp[i * K + j] = Aug[i * LD + K + j];
}

// knots at S[oX..], values at S[oY..], second derivatives at S[oM2..]
__device__ __forceinline__ double spline_eval(int oX, int oY, int oM2, int K, double x) {
    int i = 0;
    while (i + 2 < K && x >= S[oX + i + 1]) ++i;
    double h = S[oX + i + 1] - S[oX + i];
    double a = (S[oX + i + 1] - x) / h;
    double b = (x - S[oX + i]) / h;
    return a * S[oY + i] + b * S[oY + i + 1] +
           ((a * a * a - a) * S[oM2 + i] + (b * b * b - b) * S[oM2 + i + 1]) * (h * h) / 6.0;
}

template <int NS, int ME>
__global__ void __launch_bounds__(FA_WARPS * 32, 3) fa_select_kernel(FaArgs A) {
    constexpr int FA_PS = (ME < NS) ? ME : NS;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int n = A.cfg.nT2, m = A.cfg.nTE, nA = A.cfg.nA;
    Slots<NS> W;
    const int wbase = warp * fa_warp_doubles<NS>(A.pmax);
    W.carve(wbase, A.pmax);
    const int oM = wbase + Slots<NS>::doubles(A.pmax);
    const bool brute = (A.cfg.method == MET2_FA_BRUTE_FORCE);
    const int K = A.cfg.nKnots;
    double fs[NS];
#pragma unroll
    for (int s = 0; s < NS; ++s) fs[s] = 0.0;
    const long long gw = (long long)blockIdx.x * FA_WARPS + warp;
    const long long nw = (long long)gridDim.x * FA_WARPS;
    for (long long v = gw; v < A.V; v += nw) {
        unsigned st = load_signal<ME>(A.sig, v, m, oM, lane);
        if (st) {
            if (lane == 0) {
                A.fa_index[v] = 0;
                A.fa_deg[v] = 0.0;
                A.km[v] = 0.0;
                A.status[v] |= st;
            }
            continue;
        }
        int index;
        if (brute) {
            index = A.fa_index[v];
        } else {
            // knot values and second derivatives into shared scratch: gs = y, rs = Msec, xs = knots
            if (lane < K) {
                S[W.gs + lane] = A.resid[v * K + lane];
                S[W.xs + lane] = A.knots[lane];
            }
            __syncwarp();
            if (lane < K) {
                double acc = 0.0;
                for (int j = 0; j < K; ++j) acc += A.wsp[lane * K + j] * S[W.gs + j];
                S[W.rs + lane] = acc;
            }
            __syncwarp();
            Brent B;
            double xq = B.start(A.cfg.brent_lo, A.cfg.brent_hi, A.cfg.brent_xatol, A.cfg.brent_maxfun);
            while (B.feed(spline_eval(W.xs, W.gs, W.rs, K, xq), xq)) {
            }
            const double xmin = B.xf;
            // indexFA = argmin |alpha_values - res.x| (first minimum; fa_estimation.py:57)
            double bd = 1.0e300;
            int bi = -1;
            for (int i = lane; i < nA; i += 32) {
                double d = fabs(A.alphas[i] - xmin);
                if (d < bd) {
                    bd = d;
                    bi = i;
                }
            }
            double dmin;
            index = warp_argmin_nonneg(bd, bi, dmin);
            if (index < 0) index = 0;
            __syncwarp();
        }
        double kmv = 0.0;
        if (A.cfg.final_solve) {
            const double* D = A.dic + (size_t)index * m * n;
            const double* G = A.G + (size_t)index * n * n;
            compute_c<NS>(W, D, oM, m, n, lane);
            int nst = 0;
            set_dspace<NS>(W, A.dicT + (size_t)index * n * m, oM, lane);
            (void)nnls_gram<NS, false, FA_PS>(W, 0, G, n, 0, false, 0.0, n, m, lane, nst);
            if (nst && lane == 0) A.status[v] |= MET2_ST_ITMAX;
            // nnls_gram leaves the solution in column space in S[W.xc..]; km = sum(f)
            double part = 0.0;
#pragma unroll
            for (int s = 0; s < NS; ++s) {
                int col = NS * lane + s;
                double xv = (col < n) ? S[W.xc + col] : 0.0;
                fs[s] += xv;
                part += xv;
            }
            kmv = warp_sum(part);
            __syncwarp();
        }
        if (lane == 0) {
            A.fa_index[v] = index;
            A.fa_deg[v] = A.alphas[index];
            A.km[v] = kmv;
        }
    }
    if (A.partial) {
#pragma unroll
        for (int s = 0; s < NS; ++s) {
            int col = NS * lane + s;
            if (col < n) A.partial[gw * n + col] = fs[s];
        }
    }
}

// One CTA per T2 bin: thread t adds rows t, t + 256, ... and a shared-memory tree joins the 256 partial sums — a fixed
// order for a given launch geometry.  (Round 1: one thread per bin walked all ~9 500 rows, 178 us for 60 sums.)
__global__ void __launch_bounds__(256) reduce_partials_kernel(const double* __restrict__ partial, long long nrows, int n,
                                                              double* __restrict__ out) {
    __shared__ double part[256];
    const int c = blockIdx.x;
    double acc = 0.0;
    for (long long r = threadIdx.x; r < nrows; r += 256) acc += partial[r * n + c];
    part[threadIdx.x] = acc;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) part[threadIdx.x] += part[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) out[c] = part[0];
}

struct FaGeom {
    int grid;          // select kernel
    size_t smem;
    int pmax;
    int grid_search;   // search kernel: one CTA of up to FA_SEARCH_WARPS warps per SM, tables staged in shared memory
    size_t smem_search;
    int warps_search;
    int mr_thread;     // thread-per-voxel search: padded echo count (0 = not available for these sizes)
    int threads_thread, grid_thread;
    size_t smem_thread;
};

// Geometry of the thread-per-voxel search for V voxels: the largest CTA (multiple of 32 threads) whose per-thread columns
// fit beside the tables, not larger than what gives every SM a batch.  MET2_FA_SEARCH=warp switches the kernel off.
static void fa_thread_geometry(FaGeom& g, const met2_fa_cfg* cfg, long long V, int sms, const Overrides& ov) {
    g.mr_thread = 0;
    g.threads_thread = g.grid_thread = 0;
    g.smem_thread = 0;
    if (ov.fa_search_warp) return;
    // a few voxels per SM are latency bound either way and the warp kernel stages its tables with more threads
    // (config 1, 1 024 voxels: 2.4 ms with the warp kernel, 19 ms with 32-thread CTAs of this one)
    if (V < (long long)sms * 64 && !ov.fa_thread_pcap_set) return;
    const int m = cfg->nTE, n = cfg->nT2;
    const int mr = (m <= 32) ? 32 : ((m <= 48) ? 48 : 64);
    const size_t tables = sizeof(double) * (size_t)(mr == 32 ? ft_table_doubles<32>(n) : (mr == 48 ? ft_table_doubles<48>(n) : ft_table_doubles<64>(n)));
    const size_t per_thread = sizeof(double) * (size_t)ft_thread_doubles();
    const size_t budget = 227 * 1024 - 1024;
    if (tables + 64 * per_thread > budget) return;
    int t = (int)((budget - tables) / per_thread) & ~31;
    const int tmax = (mr == 32) ? FT_MAX_THREADS : FT_MAX_THREADS / 2;   // the wider residuals need the registers of two threads
    if (t > tmax) t = tmax;
    long long want = ((V + sms - 1) / sms + 31) & ~31LL;   // small batches: give every SM something to do
    if (want < 32) want = 32;
    if (t > want) t = (int)want;
    g.mr_thread = mr;
    g.threads_thread = t;
    long long nb = (V + t - 1) / t;
    g.grid_thread = (int)(nb < sms ? nb : sms);
    if (g.grid_thread < 1) g.grid_thread = 1;
    g.smem_thread = tables + per_thread * t;
}

template <int NS>
static FaGeom fa_geometry(const met2_fa_cfg* cfg, long long V, const Overrides& ov) {
    FaGeom g;
    g.pmax = cfg->nT2 < cfg->nTE ? cfg->nT2 : cfg->nTE;
    g.smem = sizeof(double) * (size_t)fa_warp_doubles<NS>(g.pmax) * FA_WARPS;
    int per_sm = (int)((size_t)(200 * 1024) / (g.smem + 1024));
    if (per_sm < 1) per_sm = 1;
    if (per_sm > 8) per_sm = 8;
    int sms = sm_count();
    if (sms <= 0) sms = 148;
    g.grid = sms * per_sm;
    g.grid_search = sms;
    {
        const size_t tables = sizeof(double) * (size_t)fa_table_doubles(cfg->nT2, cfg->nTE);
        const size_t per_warp = sizeof(double) * (size_t)fa_warp_doubles<NS>(g.pmax);
        const size_t budget = 227 * 1024 - 1024;
        int w = tables < budget ? (int)((budget - tables) / per_warp) : 0;
        if (w > FA_SEARCH_WARPS) w = FA_SEARCH_WARPS;
        if (w < 1) w = 1;
        g.warps_search = w;
        g.smem_search = tables + per_warp * w;
    }
    fa_thread_geometry(g, cfg, V, sms, ov);
    return g;
}

static FaGeom fa_geometry_any(const met2_fa_cfg* cfg, long long V, const Overrides& ov) {
    int ns = (cfg->nT2 + 31) / 32;
    if (ns <= 2) return fa_geometry<2>(cfg, V, ov);
    if (ns == 3) return fa_geometry<3>(cfg, V, ov);
    return fa_geometry<4>(cfg, V, ov);
}

template <int MR>
static int fa_launch_thread(const FaArgs& A, const FaGeom& g, cudaStream_t st) {
    cudaError_t e = cudaFuncSetAttribute(fa_search_thread_kernel<MR>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)g.smem_thread);
    if (e != cudaSuccess) return set_error(MET2_ERR_CUDA, "fa_search_thread attr: %s", cudaGetErrorString(e));
    MET2_LAUNCH(g.grid_thread, g.threads_thread, g.smem_thread, st, fa_search_thread_kernel<MR>)(A);
    count_launch();
    return check_launch("fa_search_thread_kernel");
}

template <int NS, int ME>
static int fa_launch(const FaArgs& A, const FaGeom& g, cudaStream_t st) {
    cudaError_t e;
    e = cudaFuncSetAttribute(fa_search_kernel<NS, ME>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             (int)g.smem_search);
    if (e != cudaSuccess) return set_error(MET2_ERR_CUDA, "fa_search attr: %s", cudaGetErrorString(e));
    e = cudaFuncSetAttribute(fa_select_kernel<NS, ME>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)g.smem);
    if (e != cudaSuccess) return set_error(MET2_ERR_CUDA, "fa_select attr: %s", cudaGetErrorString(e));
    int rc;
    FaArgs B = A;
    if (g.mr_thread) {
        // thread per voxel first; the warp-per-voxel kernel then redoes the voxels it handed back (usually none)
        e = cudaMemsetAsync(A.ovf_count, 0, sizeof(int), st);
        if (e != cudaSuccess) return set_error(MET2_ERR_CUDA, "memset ovf_count: %s", cudaGetErrorString(e));
        rc = (g.mr_thread == 32) ? fa_launch_thread<32>(A, g, st)
                                 : ((g.mr_thread == 48) ? fa_launch_thread<48>(A, g, st) : fa_launch_thread<64>(A, g, st));
        if (rc) return rc;
        B.vlist = A.ovf_list;
    }
    MET2_LAUNCH(g.grid_search, g.warps_search * 32, g.smem_search, st, fa_search_kernel<NS, ME>)(B);
    count_launch();
    rc = check_launch("fa_search_kernel");
    if (rc) return rc;
    if (A.cfg.method == MET2_FA_SPLINE) {
        MET2_LAUNCH(1, 32, 0, st, spline_weights_kernel)(A.knots, A.cfg.nKnots, A.wsp);
        count_launch();
        rc = check_launch("spline_weights_kernel");
        if (rc) return rc;
    }
    MET2_LAUNCH(g.grid, FA_WARPS * 32, g.smem, st, fa_select_kernel<NS, ME>)(A);
    count_launch();
    rc = check_launch("fa_select_kernel");
    if (rc) return rc;
    if (A.fsol_sum) {
        MET2_LAUNCH(A.cfg.nT2, 256, 0, st, reduce_partials_kernel)(A.partial, (long long)g.grid * FA_WARPS, A.cfg.nT2,
                                                                   A.fsol_sum);
        count_launch();
        rc = check_launch("reduce_partials_kernel");
    }
    return rc;
}

}  // namespace met2

using namespace met2;

static int fa_check_cfg(const met2_fa_cfg* cfg) {
    if (!cfg) return set_error(MET2_ERR_ARG, "met2_fa: cfg is NULL");
    if (cfg->nT2 <= 0 || cfg->nT2 > MET2_MAX_NT2 || cfg->nTE <= 0 || cfg->nTE > MET2_MAX_NTE || cfg->nA <= 0)
        return set_error(MET2_ERR_ARG, "met2_fa: unsupported sizes nT2=%d nTE=%d nA=%d", cfg->nT2, cfg->nTE, cfg->nA);
    if (cfg->method != MET2_FA_BRUTE_FORCE && cfg->method != MET2_FA_SPLINE)
        return set_error(MET2_ERR_ARG, "met2_fa: unknown method %d", cfg->method);
    if (cfg->method == MET2_FA_SPLINE && (cfg->nKnots < 4 || cfg->nKnots > MET2_MAX_KNOTS))
        return set_error(MET2_ERR_ARG, "met2_fa: spline needs 4..%d knots, got %d", MET2_MAX_KNOTS, cfg->nKnots);
    return MET2_OK;
}

extern "C" int64_t met2_fa_workspace_bytes(int64_t V, const met2_fa_cfg* cfg) {
    if (fa_check_cfg(cfg) || V < 0) return -1;
    FaGeom g = fa_geometry_any(cfg, V, read_overrides());
    int nS = cfg->method == MET2_FA_SPLINE ? cfg->nKnots : 1;
    size_t b = align256(sizeof(double) * (size_t)V * nS);
    b += align256(sizeof(double) * MET2_MAX_KNOTS * MET2_MAX_KNOTS);
    b += align256(sizeof(double) * (size_t)g.grid * FA_WARPS * cfg->nT2);
    b += align256(sizeof(int) * (size_t)V) + align256(sizeof(int) * (size_t)V * FA_CARRY) +
         align256(sizeof(double) * (size_t)V * FA_CARRY);
    b += align256(sizeof(int) * (size_t)V) + 256;   // ovf_list, ovf_count
    return (int64_t)b + 256;
}

extern "C" int met2_fa_fit(const double* sig, int64_t V, const met2_fa_cfg* cfg, const double* dic, const double* dicT,
                           const double* G, const double* alphas, const double* dic_s, const double* dicT_s,
                           const double* G_s, const double* knots, int32_t* fa_index, double* fa_deg, double* km,
                           double* fsol_sum, uint32_t* status, void* workspace, void* stream) {
    int rc = fa_check_cfg(cfg);
    if (rc) return rc;
    if (V < 0 || !sig || !dic || !dicT || !G || !alphas || !fa_index || !fa_deg || !km || !status || !workspace)
        return set_error(MET2_ERR_ARG, "met2_fa_fit: NULL argument");
    const bool spline = cfg->method == MET2_FA_SPLINE;
    if (spline && (!dic_s || !dicT_s || !G_s || !knots))
        return set_error(MET2_ERR_ARG, "met2_fa_fit: spline method needs the coarse dictionary and knots");
    if (V == 0) return MET2_OK;
    cudaStream_t st = (cudaStream_t)stream;
    const Overrides ov = read_overrides();
    FaGeom g = fa_geometry_any(cfg, V, ov);
    FaArgs A;
    A.sig = sig;
    A.V = V;
    A.cfg = *cfg;
    A.dic = dic; A.dicT = dicT; A.G = G; A.alphas = alphas;
    if (spline) {
        A.dic_s = dic_s; A.dicT_s = dicT_s; A.G_s = G_s; A.knots = knots;
        A.nS = cfg->nKnots;
    } else {
        A.dic_s = dic; A.dicT_s = dicT; A.G_s = G; A.knots = nullptr;
        A.nS = cfg->nA;
    }
    A.fa_index = fa_index; A.fa_deg = fa_deg; A.km = km; A.fsol_sum = fsol_sum; A.status = status;
    unsigned char* w = reinterpret_cast<unsigned char*>(((uintptr_t)workspace + 255) & ~(uintptr_t)255);
    int nSr = spline ? cfg->nKnots : 1;
    A.resid = reinterpret_cast<double*>(w);
    w += align256(sizeof(double) * (size_t)V * nSr);
    A.wsp = reinterpret_cast<double*>(w);
    w += align256(sizeof(double) * MET2_MAX_KNOTS * MET2_MAX_KNOTS);
    A.partial = fsol_sum ? reinterpret_cast<double*>(w) : nullptr;
    w += align256(sizeof(double) * (size_t)g.grid * FA_WARPS * cfg->nT2);
    A.ws_p = reinterpret_cast<int*>(w);
    w += align256(sizeof(int) * (size_t)V);
    A.ws_ix = reinterpret_cast<int*>(w);
    w += align256(sizeof(int) * (size_t)V * FA_CARRY);
    A.ws_x = reinterpret_cast<double*>(w);
    w += align256(sizeof(double) * (size_t)V * FA_CARRY);
    A.ovf_list = reinterpret_cast<int*>(w);
    w += align256(sizeof(int) * (size_t)V);
    A.ovf_count = reinterpret_cast<int*>(w);
    A.vlist = nullptr;
    A.thread_pcap = FT_PM;
    if (ov.fa_thread_pcap >= 1 && ov.fa_thread_pcap < FT_PM) A.thread_pcap = ov.fa_thread_pcap;
    A.pmax = g.pmax;
    cudaError_t e = cudaMemsetAsync(status, 0, sizeof(uint32_t) * (size_t)V, st);
    if (e != cudaSuccess) return set_error(MET2_ERR_CUDA, "memset status: %s", cudaGetErrorString(e));
    int ns = (cfg->nT2 + 31) / 32;
    int me = (cfg->nTE + 31) / 32;
    if (ns <= 2 && me == 1) return fa_launch<2, 1>(A, g, st);
    if (ns <= 2 && me == 2) return fa_launch<2, 2>(A, g, st);
    if (ns == 3 && me == 1) return fa_launch<3, 1>(A, g, st);
    if (ns == 3 && me == 2) return fa_launch<3, 2>(A, g, st);
    if (ns == 4 && me == 1) return fa_launch<4, 1>(A, g, st);
    if (ns == 4 && me == 2) return fa_launch<4, 2>(A, g, st);
    return set_error(MET2_ERR_UNSUPPORTED, "met2_fa_fit: unsupported template sizes");
}
