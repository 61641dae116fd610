// met2_param.cu — three-pool parametric T2 fit (no counterpart in the reference): bounded Levenberg-Marquardt over
// three discrete EPG pools that share one continuous refocusing angle (met2_param_fit).
//
// Definition (tests/param_oracle.py restates it in NumPy line for line; DESIGN.md §10c).  Normalised units like the
// point fit: y = sig / sig[0].  Inputs are the point fit's outputs; voxels whose status has MET2_ST_SKIPPED or
// MET2_ST_NONFINITE are not fitted and get all-zero outputs (status: those bits).
//   d(T2, alpha)[e]  = the column met2_epg_dictionary produces for (alpha, T2): epg_decay's recurrence (met2_epg.cuh),
//                      excitation alpha/2, scaled by (1 - exp(-TR/T1)), with cfg's T1 and tau.
//   m(p)             = A_m d(T2_m, alpha) + A_ie d(T2_ie, alpha) + A_fw d(T2_fw, alpha)   (summed in that order)
//   p                = (A_m, A_ie, A_fw, u_m, u_ie, u_fw, alpha),  u = ln T2 (ms),  alpha in degrees
//   box              A_c >= 0,  T2_c in [t2_lo[c], t2_hi[c]] (u in [ln t2_lo, ln t2_hi]),  alpha in [fa_lo, fa_hi]
//                    (batched.Met2Plan: T2s[0] / myelin_T2 / 200 / T2s[-1] and 90 / 180, motor...:215-220)
//   start            x = fsol / sig[0];  A_c = sum of x_j over the bins with comp bit c;  u_c = the x-weighted mean of
//                    ln T2_j over those bins, clipped into its box, or the midpoint of the u box when A_c = 0;
//                    alpha = fa_deg clipped into its box
//   cost             F = 1/2 ||m(p) - y||^2
//   J = dm/dp        forward-mode: every state of the recurrence carries d/du and d/dalpha (met2::Dual below), the
//                    initial state sin(alpha/2), cos(alpha/2) included.  J_{A_c} = d_c, J_{u_c} = A_c dd_c/du,
//                    J_alpha = sum_c A_c dd_c/dalpha.  g = J^T r, H = J^T J, r = m - y.
//   projected LM     it = 0, mu = mu0; at the start point F, g, H.  Repeat:
//                      1. it == max_iter: MET2_ST_ITMAX, stop.   it += 1.
//                      2. free set: i is free unless H_ii == 0 (a zero J column: the u_c of a pool with A_c = 0), or
//                         p_i == lo_i and g_i > 0, or p_i == hi_i and g_i < 0.  No free variable: stop.
//                      3. Cholesky of M = H_FF + mu diag(H_FF) (7 x 7 at most; the rows of the other variables are
//                         the identity and their right-hand side 0).  A pivot <= 0 (or NaN): mu *= 10, stop if
//                         mu > mu_max, else next iteration.  delta = -M^{-1} g.
//                      4. t = clip(p + delta, lo, hi).  ||t - p|| <= xtol (xtol + ||p||): stop.
//                      5. F_t, g_t, H_t at t.  F_t < F: accept (p = t, ...), mu /= 10, stop if (F - F_t) <= ftol F.
//                         Otherwise mu *= 10, stop if mu > mu_max.
//                    Defaults (batched.PARAM_DEFAULTS): mu0 1e-3, mu_max 1e16, ftol 1e-12, xtol 1e-10, max_iter 2000
//                    (the fit creeps along flat valleys: noiseless three-pool voxels need up to ~1 600 iterations).
//   outputs (raw units)
//                    params [V][7] = A_c sig[0] (3), exp(u_c) (3, ms), alpha;  maps [V][6] = MWF, IEWF, FWF = A_c / sum A
//                    (0 when sum A = 0), T2_M = exp(u_m), T2_IE = exp(u_ie) (0 when that pool's A is 0),
//                    TWC = sig[0] sum A;  est_signal [V][nTE] = sig[0] m(p);  sse [V] = sig[0]^2 ||m - y||^2;
//                    iters [V] = it;  status [V] = the input's MET2_ST_SKIPPED | MET2_ST_NONFINITE bits, MET2_ST_ITMAX,
//                    and MET2_ST_AT_BOUND when a u_c or alpha ends on its box (informational).
//
// Layout: one warp per voxel, 4 voxels per block, no block barrier.  Lane l holds the EPG states k = l + 1 + 32 s
// (s < ME slots, ME = 2 for nTE > 32) as Duals; the shifts of F+k up and F-k down are __shfl_sync, F0 is broadcast from
// lane 0, and states k > nTE are held at zero so the truncation matches epg_decay's.  Lane l also owns echoes
// e = l + 32 s, where it keeps m and the J row; H, g and F are butterfly sums (every lane gets the same bits), and
// every lane runs the 7 x 7 Cholesky redundantly, so the LM control flow is warp-uniform.
#include <math.h>

#include "met2_host.h"
#include "met2_epg.cuh"

namespace met2 {

constexpr int PF_WARPS = 4;   // voxels per block
constexpr int PF_NP = 7;      // parameters
constexpr int PF_NH = PF_NP * (PF_NP + 1) / 2;

// A value with its derivatives with respect to u = ln T2 and alpha (deg).  Each operation rounds its value part exactly
// like the double operation it replaces, so the EPG recurrence of met2_epg.cuh gives the dictionary's values.
struct Dual {
    double v, t, a;
};
__device__ __forceinline__ Dual operator+(Dual x, Dual y) { return {x.v + y.v, x.t + y.t, x.a + y.a}; }
__device__ __forceinline__ Dual operator-(Dual x, Dual y) { return {x.v - y.v, x.t - y.t, x.a - y.a}; }
__device__ __forceinline__ Dual operator*(Dual x, Dual y) {
    return {x.v * y.v, x.t * y.v + x.v * y.t, x.a * y.v + x.v * y.a};
}
__device__ __forceinline__ Dual operator*(Dual x, double s) { return {x.v * s, x.t * s, x.a * s}; }
__device__ __forceinline__ Dual operator*(double s, Dual x) { return {s * x.v, s * x.t, s * x.a}; }
__device__ __forceinline__ Dual operator/(Dual x, double s) { return {x.v / s, x.t / s, x.a / s}; }
__device__ __forceinline__ Dual operator/(double s, Dual x) {
    const double r = s / x.v, d = -r / x.v;
    return {r, d * x.t, d * x.a};
}
__device__ __forceinline__ Dual exp(Dual x) {
    const double e = ::exp(x.v);
    return {e, e * x.t, e * x.a};
}
__device__ __forceinline__ Dual sin(Dual x) {
    const double s = ::sin(x.v), c = ::cos(x.v);
    return {s, c * x.t, c * x.a};
}
__device__ __forceinline__ Dual cos(Dual x) {
    const double s = ::sin(x.v), c = ::cos(x.v);
    return {c, -s * x.t, -s * x.a};
}
__device__ __forceinline__ Dual shfl(Dual x, int src) {
    return {__shfl_sync(0xffffffffu, x.v, src), __shfl_sync(0xffffffffu, x.t, src), __shfl_sync(0xffffffffu, x.a, src)};
}

__device__ __forceinline__ double warp_sum(double v) {
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

struct PfArgs {
    const double* sig;        // [V][m]
    const double* fa_deg;     // [V]
    const double* fsol;       // [V][n]
    const uint32_t* status_in;
    const double* logT2;      // [n]
    const uint8_t* comp;      // [n]
    long long V;
    int m, n, max_iter;
    double tau, TR, T1;
    double lo[PF_NP], hi[PF_NP];
    double mu0, mu_max, ftol, xtol;
    double *params, *maps, *est, *sse;
    int32_t* iters;
    uint32_t* status;
};

// One pool's decay curve d(T2, alpha) and its derivatives at the echoes e = lane + 32 s this lane owns.
template <int ME>
__device__ __forceinline__ void pool_curve(const PfArgs& A, double u, double alpha, int lane, Dual d[ME]) {
    const double T2 = ::exp(u);
    const EpgCoef<Dual> c = epg_coef(Dual{alpha, 0.0, 1.0}, Dual{T2, T2, 0.0}, A.T1, A.tau);
    const double scale = 1.0 - ::exp(-A.TR / A.T1);   // epg_dictionary_kernel's scale
    const Dual zero = {0.0, 0.0, 0.0};
    Dual fp[ME], fm[ME], z[ME];
#pragma unroll
    for (int s = 0; s < ME; ++s) {
        fp[s] = fm[s] = z[s] = zero;
        d[s] = zero;
    }
    Dual F0 = c.f0;
    if (lane == 0) fm[0] = c.fm1;
    const int n = A.m;
    for (int echo = 0; echo < n; ++echo) {
        for (int half_step = 0; half_step < 2; ++half_step) {
            // shift: F0 <- F-1, F+k <- F+(k-1) (F+1 <- F0), F-k <- F-(k+1)
            const Dual newF0 = shfl(fm[0], 0);
            Dual up[ME], dn[ME];
#pragma unroll
            for (int s = 0; s < ME; ++s) {
                up[s] = shfl(fp[s], (lane + 31) & 31);
                dn[s] = shfl(fm[s], (lane + 1) & 31);
            }
#pragma unroll
            for (int s = 0; s < ME; ++s) {
                fp[s] = lane ? up[s] : (s == 0 ? F0 : up[s - 1]);
                fm[s] = lane < 31 ? dn[s] : (s + 1 < ME ? dn[s + 1] : zero);
                if (lane + 1 + 32 * s > n) fp[s] = fm[s] = z[s] = zero;
            }
            F0 = newF0 * c.e2;
#pragma unroll
            for (int s = 0; s < ME; ++s) epg_relax(fp[s], fm[s], z[s], c);
            if (half_step == 0) {
#pragma unroll
                for (int s = 0; s < ME; ++s) epg_rf(fp[s], fm[s], z[s], c);
            }
        }
#pragma unroll
        for (int s = 0; s < ME; ++s)
            if (echo == lane + 32 * s) d[s] = scale * F0;
    }
}

// Model, residual sums and normal equations at p: m [ME] per lane; F, g [7], H [28] (packed lower) on every lane.
template <int ME>
__device__ void evaluate(const PfArgs& A, const double p[PF_NP], const double y[ME], int lane, double m[ME], double& F,
                         double g[PF_NP], double H[PF_NH]) {
    Dual d0[ME], d1[ME], d2[ME];
    pool_curve<ME>(A, p[3], p[6], lane, d0);
    pool_curve<ME>(A, p[4], p[6], lane, d1);
    pool_curve<ME>(A, p[5], p[6], lane, d2);
    double f = 0.0, gl[PF_NP], Hl[PF_NH];
#pragma unroll
    for (int i = 0; i < PF_NP; ++i) gl[i] = 0.0;
#pragma unroll
    for (int i = 0; i < PF_NH; ++i) Hl[i] = 0.0;
#pragma unroll
    for (int s = 0; s < ME; ++s) {
        m[s] = 0.0;
        if (lane + 32 * s >= A.m) continue;
        m[s] = p[0] * d0[s].v + p[1] * d1[s].v + p[2] * d2[s].v;
        const double r = m[s] - y[s];
        const double J[PF_NP] = {d0[s].v,        d1[s].v,        d2[s].v,
                                 p[0] * d0[s].t, p[1] * d1[s].t, p[2] * d2[s].t,
                                 p[0] * d0[s].a + p[1] * d1[s].a + p[2] * d2[s].a};
        f += r * r;
        int k = 0;
#pragma unroll
        for (int i = 0; i < PF_NP; ++i) {
            gl[i] += J[i] * r;
#pragma unroll
            for (int j = 0; j <= i; ++j) Hl[k++] += J[i] * J[j];
        }
    }
    F = 0.5 * warp_sum(f);
#pragma unroll
    for (int i = 0; i < PF_NP; ++i) g[i] = warp_sum(gl[i]);
#pragma unroll
    for (int i = 0; i < PF_NH; ++i) H[i] = warp_sum(Hl[i]);
}

__device__ __forceinline__ int hidx(int i, int j) { return i * (i + 1) / 2 + j; }   // i >= j

template <int ME>
__global__ void __launch_bounds__(PF_WARPS * 32) param_fit_kernel(PfArgs A) {
    const int lane = threadIdx.x & 31;
    const long long v = (long long)blockIdx.x * PF_WARPS + (threadIdx.x >> 5);
    if (v >= A.V) return;
    const int m = A.m, n = A.n;
    const double* sig = A.sig + v * m;
    const uint32_t st_in = A.status_in[v] & (MET2_ST_SKIPPED | MET2_ST_NONFINITE);
    if (st_in) {
        for (int i = lane; i < PF_NP; i += 32) A.params[v * PF_NP + i] = 0.0;
        for (int i = lane; i < 6; i += 32) A.maps[v * 6 + i] = 0.0;
        for (int e = lane; e < m; e += 32) A.est[v * m + e] = 0.0;
        if (lane == 0) {
            A.sse[v] = 0.0;
            A.iters[v] = 0;
            A.status[v] = st_in;
        }
        return;
    }
    const double s0 = sig[0];
    double y[ME];
#pragma unroll
    for (int s = 0; s < ME; ++s) y[s] = lane + 32 * s < m ? sig[lane + 32 * s] / s0 : 0.0;

    // start from the point fit's spectrum
    double p[PF_NP];
    {
        double Ac[3] = {0.0, 0.0, 0.0}, Wc[3] = {0.0, 0.0, 0.0};
        for (int j = lane; j < n; j += 32) {
            const double x = A.fsol[v * n + j] / s0;
            const uint8_t cj = A.comp[j];
#pragma unroll
            for (int c = 0; c < 3; ++c)
                if (cj & (1u << c)) {
                    Ac[c] += x;
                    Wc[c] += x * A.logT2[j];
                }
        }
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const double a = warp_sum(Ac[c]), w = warp_sum(Wc[c]);
            p[c] = a;
            const double u = a > 0.0 ? w / a : 0.5 * (A.lo[3 + c] + A.hi[3 + c]);
            p[3 + c] = fmin(fmax(u, A.lo[3 + c]), A.hi[3 + c]);
        }
        p[6] = fmin(fmax(A.fa_deg[v], A.lo[6]), A.hi[6]);
    }

    double mc[ME], F, g[PF_NP], H[PF_NH];
    evaluate<ME>(A, p, y, lane, mc, F, g, H);
    double mu = A.mu0;
    int it = 0;
    uint32_t st = 0;
    for (;;) {
        if (it == A.max_iter) {
            st |= MET2_ST_ITMAX;
            break;
        }
        ++it;
        bool fr[PF_NP];
        int nfree = 0;
#pragma unroll
        for (int i = 0; i < PF_NP; ++i) {
            fr[i] = !(H[hidx(i, i)] == 0.0 || (p[i] <= A.lo[i] && g[i] > 0.0) || (p[i] >= A.hi[i] && g[i] < 0.0));
            nfree += fr[i];
        }
        if (nfree == 0) break;
        // Cholesky of M = H_FF + mu diag(H_FF), identity rows elsewhere; delta = -M^{-1} g
        double L[PF_NH], b[PF_NP];
        bool pd = true;
#pragma unroll
        for (int i = 0; i < PF_NP; ++i) {
#pragma unroll
            for (int j = 0; j <= i; ++j) {
                double mij;
                if (i == j) mij = fr[i] ? H[hidx(i, i)] + mu * H[hidx(i, i)] : 1.0;
                else mij = fr[i] && fr[j] ? H[hidx(i, j)] : 0.0;
                for (int k = 0; k < j; ++k) mij -= L[hidx(i, k)] * L[hidx(j, k)];
                if (i == j) {
                    pd = pd && mij > 0.0;
                    L[hidx(i, i)] = sqrt(mij);
                } else {
                    L[hidx(i, j)] = mij / L[hidx(j, j)];
                }
            }
        }
        if (!pd) {
            mu *= 10.0;
            if (mu > A.mu_max) break;
            continue;
        }
#pragma unroll
        for (int i = 0; i < PF_NP; ++i) {
            double s = fr[i] ? -g[i] : 0.0;
            for (int k = 0; k < i; ++k) s -= L[hidx(i, k)] * b[k];
            b[i] = s / L[hidx(i, i)];
        }
#pragma unroll
        for (int i = PF_NP - 1; i >= 0; --i) {
            double s = b[i];
            for (int k = i + 1; k < PF_NP; ++k) s -= L[hidx(k, i)] * b[k];
            b[i] = s / L[hidx(i, i)];
        }
        double t[PF_NP], dn = 0.0, pn = 0.0;
#pragma unroll
        for (int i = 0; i < PF_NP; ++i) {
            t[i] = fr[i] ? fmin(fmax(p[i] + b[i], A.lo[i]), A.hi[i]) : p[i];
            dn += (t[i] - p[i]) * (t[i] - p[i]);
            pn += p[i] * p[i];
        }
        if (sqrt(dn) <= A.xtol * (A.xtol + sqrt(pn))) break;
        double mt[ME], Ft, gt[PF_NP], Ht[PF_NH];
        evaluate<ME>(A, t, y, lane, mt, Ft, gt, Ht);
        if (Ft < F) {
            const bool done = F - Ft <= A.ftol * F;
#pragma unroll
            for (int i = 0; i < PF_NP; ++i) {
                p[i] = t[i];
                g[i] = gt[i];
            }
#pragma unroll
            for (int i = 0; i < PF_NH; ++i) H[i] = Ht[i];
#pragma unroll
            for (int s = 0; s < ME; ++s) mc[s] = mt[s];
            F = Ft;
            mu /= 10.0;
            if (done) break;
        } else {
            mu *= 10.0;
            if (mu > A.mu_max) break;
        }
    }

    for (int i = 3; i < PF_NP; ++i)
        if (p[i] == A.lo[i] || p[i] == A.hi[i]) st |= MET2_ST_AT_BOUND;
#pragma unroll
    for (int s = 0; s < ME; ++s)
        if (lane + 32 * s < m) A.est[v * m + lane + 32 * s] = s0 * mc[s];
    if (lane == 0) {
        const double sumA = p[0] + p[1] + p[2];
        double* P = A.params + v * PF_NP;
        double* M = A.maps + v * 6;
        for (int c = 0; c < 3; ++c) {
            P[c] = p[c] * s0;
            P[3 + c] = ::exp(p[3 + c]);
            M[c] = sumA > 0.0 ? p[c] / sumA : 0.0;
        }
        P[6] = p[6];
        M[3] = p[0] > 0.0 ? P[3] : 0.0;
        M[4] = p[1] > 0.0 ? P[4] : 0.0;
        M[5] = s0 * sumA;
        A.sse[v] = (s0 * s0) * (2.0 * F);
        A.iters[v] = it;
        A.status[v] = st;
    }
}

}  // namespace met2

using namespace met2;

extern "C" int met2_param_fit(const double* sig, const double* fa_deg, const double* fsol, const uint32_t* status_in,
                              int64_t V, const met2_param_cfg* cfg, const double* logT2, const uint8_t* comp,
                              double* params, double* maps, double* est_signal, double* sse, int32_t* iters,
                              uint32_t* status, void* stream) {
    if (!cfg || V < 0 || V >= (int64_t)1 << 31)
        return set_error(MET2_ERR_ARG, "met2_param_fit: bad argument (cfg=%p, V=%lld)", (const void*)cfg, (long long)V);
    const met2_param_cfg& c = *cfg;
    if (c.nTE <= 0 || c.nTE > MET2_MAX_NTE || c.nT2 <= 0 || c.nT2 > MET2_MAX_NT2 || c.max_iter < 0)
        return set_error(MET2_ERR_ARG, "met2_param_fit: bad sizes (nTE=%d nT2=%d max_iter=%d)", c.nTE, c.nT2,
                         c.max_iter);
    if (!(c.tau > 0.0) || !isfinite(c.tau) || !(c.T1 > 0.0) || !isfinite(c.T1) || !isfinite(c.TR))
        return set_error(MET2_ERR_ARG, "met2_param_fit: bad timing (tau=%g TR=%g T1=%g)", c.tau, c.TR, c.T1);
    for (int k = 0; k < 3; ++k)
        if (!(c.t2_lo[k] > 0.0) || !(c.t2_lo[k] <= c.t2_hi[k]) || !isfinite(c.t2_hi[k]))
            return set_error(MET2_ERR_ARG, "met2_param_fit: empty T2 box %d [%g, %g]", k, c.t2_lo[k], c.t2_hi[k]);
    if (!(c.fa_lo <= c.fa_hi) || !isfinite(c.fa_lo) || !isfinite(c.fa_hi))
        return set_error(MET2_ERR_ARG, "met2_param_fit: empty flip-angle box [%g, %g]", c.fa_lo, c.fa_hi);
    if (!(c.mu0 > 0.0) || !(c.mu_max >= c.mu0) || !isfinite(c.mu_max) || !(c.ftol >= 0.0) || !(c.xtol >= 0.0))
        return set_error(MET2_ERR_ARG, "met2_param_fit: bad tolerances");
    if (V > 0 && (!sig || !fa_deg || !fsol || !status_in || !logT2 || !comp || !params || !maps || !est_signal ||
                  !sse || !iters || !status))
        return set_error(MET2_ERR_ARG, "met2_param_fit: NULL argument");
    if (V == 0) return MET2_OK;
    PfArgs A;
    A.sig = sig; A.fa_deg = fa_deg; A.fsol = fsol; A.status_in = status_in; A.logT2 = logT2; A.comp = comp;
    A.V = V; A.m = c.nTE; A.n = c.nT2; A.max_iter = c.max_iter;
    A.tau = c.tau; A.TR = c.TR; A.T1 = c.T1;
    for (int k = 0; k < 3; ++k) {
        A.lo[k] = 0.0;
        A.hi[k] = INFINITY;
        A.lo[3 + k] = log(c.t2_lo[k]);
        A.hi[3 + k] = log(c.t2_hi[k]);
    }
    A.lo[6] = c.fa_lo;
    A.hi[6] = c.fa_hi;
    A.mu0 = c.mu0; A.mu_max = c.mu_max; A.ftol = c.ftol; A.xtol = c.xtol;
    A.params = params; A.maps = maps; A.est = est_signal; A.sse = sse; A.iters = iters; A.status = status;
    cudaStream_t st = (cudaStream_t)stream;
    const unsigned blocks = (unsigned)((V + PF_WARPS - 1) / PF_WARPS);
    if (c.nTE <= 32) MET2_LAUNCH(blocks, PF_WARPS * 32, 0, st, param_fit_kernel<1>)(A);
    else MET2_LAUNCH(blocks, PF_WARPS * 32, 0, st, param_fit_kernel<2>)(A);
    count_launch();
    return check_launch("met2_param_fit");
}
