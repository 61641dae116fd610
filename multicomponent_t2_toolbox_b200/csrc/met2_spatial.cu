// met2_spatial.cu — spatially regularised spectrum fitting (no counterpart in the reference): neighbour-coupled NNLS
// block updates in red-black order (met2_spatial_sweep) and the outputs of the coupled fit (met2_spatial_finish).
// The caller runs the point fit (met2_t2_fit) first; nothing here selects lambda.
//
// Definition (tests/spatial_oracle.py restates it in NumPy; DESIGN.md §10b).  All quantities are in the reference's
// normalised units.  For a fitted voxel v of the point fit (status without MET2_ST_SKIPPED):
//   y_v = sig_v / sig_v[0],  x_v = fsol_v / sig_v[0] (motor...:127-131, 153),  a_v = fa_index[v],
//   lambda_v = the lambda the point fit selected (reg under MET2_T2_FLAG_REG_IS_LAMBDA: 0 for NNLS, 1.8 for T2SPARC,
//   the selected lambda for X2, L-curve, GCV and BayesReg),  L / K = L^T L the plan's regularisation matrix,
//   N(v) = the fitted 6-connected face neighbours of v in the volume, n_v = |N(v)|.
// Joint objective, mu >= 0 given by the user, x >= 0:
//   J(x) = sum_v ||D_{a_v} x_v - y_v||^2 + lambda_v ||L x_v||^2  +  mu sum_{edges {v,n}} ||x_v - x_n||^2
// Block update of v with its neighbours held fixed, p_v = mean_{n in N(v)} x_n:
//   x_v <- argmin_{x >= 0} ||D x - y_v||^2 + lambda_v ||L x||^2 + mu n_v ||x - p_v||^2
//   Gram form: G_a + lambda_v K + mu n_v I with c = D_a^T y_v + mu n_v p_v;
//   stacked form: A = [D; sqrt(lambda_v) L; sqrt(mu n_v) I], b = [y_v; 0; sqrt(mu n_v) p_v].  n_v = 0: the point problem.
// Order: red-black.  The colour of voxel (i, j, k) is (i + j + k) mod 2; a sweep updates every colour-0 voxel, then
// every colour-1 voxel.  No face neighbour shares a voxel's colour, so a half-sweep is one launch that updates x in
// place without races, and its result does not depend on voxel order, chunking or slabs.  Each half-sweep is an exact
// block minimisation of the convex J, so J does not increase.  x^0 = fsol / sig[0] (the point fit); n_sweeps sweeps.
// Outputs: fsol = x sig[0], est_signal = D_a x sig[0], the six maps as met2_t2_fit computes them (motor...:443-472);
// FA, FA_index and reg stay the point fit's; status is the point fit's, OR'd with MET2_ST_ITMAX when a sweep solve hits
// itmax.
//
// met2_spatial_sweep: one warp per voxel of one colour's index list.  The warp gathers the <= 6 neighbour rows of x
// (lanes over T2 bins), forms c and its own band lambda_v K + mu n_v I (5-band form, passed to nnls_gram with weight 1)
// and calls the Gram-domain Lawson-Hanson of met2_nnls.cuh warm-started from the voxel's current support and
// coefficients.  The minimiser of the strictly convex block problem does not depend on the start.
//   * The D-space candidate test of nnls_gram (set_dspace) is switched OFF.  It exists for the plain problem, where
//     rho^2 = G_jj - r.r can fall below rounding; nnls_gram never runs it for a regularised solve, and every solve here
//     passes a band.  With mu n_v > 0 the band adds mu n_v to the diagonal, so rho^2 >= mu n_v.  The only plain case
//     left is an isolated voxel of an NNLS fit (lambda_v = 0, n_v = 0), whose solve starts at its own point fit.
//   * The refinement step on the final support is INCLUDED, with the prior term: refine_on_support of met2_device.cuh
//     assumes c = D^T y - lambda K x, so this file has its own step with the gradient
//     g = D_P^T (y - D_P x) - (lambda_v K x)_P - mu n_v (x - p)_P.  The Gram-domain solve loses up to ~1e-9 relative in
//     the worst Tikhonov voxels (met2_device.cuh); one step in D-space brings the block solution to ~1e-12, which is
//     what makes half-sweeps comparable with the QR-based restatement at 1e-9.
// met2_spatial_finish: one warp per voxel of the whole list: fsol, est_signal and the maps of the current x, with the
// epilogue of met2_t2_impl.cuh restated here (skipped voxels get that epilogue's zeros).
#include <math.h>

#include "met2_device.cuh"
#include "met2_host.h"

namespace met2 {

constexpr int SP_MAX_WARPS = 4;   // voxels per block (no block-wide barrier: warps retire independently)

struct SpArgs {
    const double* sig;          // [V][m] raw signals
    const int32_t* fa_index;    // [V]
    const double* lam;          // [V] lambda_v
    const int32_t* nbr;         // [V][6] neighbour positions, -1 = none
    const int32_t* vox;         // [Vc] voxels of this half-sweep
    long long V, Vc;
    int m, n, nA;
    const double *G, *dicT, *kband;
    double mu;
    double* x;                  // [V][n] normalised spectra, updated in place
    uint32_t* status;           // [V]
};

// per-warp shared memory: [NNLS slots (pmax = n)][signal 64][band 5n][prior term n]
template <int NS>
__host__ __device__ __forceinline__ int sp_warp_doubles(int n) {
    return (Slots<NS>::doubles(n) + 64 + 6 * n + 31) & ~31;
}

// One step of iterative refinement on the final support with the prior term (see the header): r = y - D_P x,
// g = D_P^T r - (Kb x)_P + cp_P, x += T T^T g, skipped if a coefficient would become non-positive.  Kb = the warp's
// band lambda_v K + mu n_v I at S[oKb + d*n + c]; cp = mu n_v p at S[oCp ..]; x in column space in S[W.xc ..].
template <int NS, int ME>
__device__ __forceinline__ void refine_prior(const Slots<NS>& W, const double* __restrict__ Dt, int oM, int m, int p,
                                             int lane, int oKb, int oCp, int n) {
    static_assert(ME <= NS, "the residual is staged in a position-space slot");
    double fit[ME];
    (void)fit_and_sse<NS, ME>(W, Dt, oM, m, p, lane, fit);
    const int oR = W.rs;
#pragma unroll
    for (int u = 0; u < ME; ++u) {
        const int e = lane + 32 * u;
        if (e < m) S[oR + e] = S[oM + e] - fit[u];
    }
    __syncwarp();
    double gv[NS];
#pragma unroll
    for (int t = 0; t < NS; ++t) {
        const int i = lane + 32 * t;
        gv[t] = 0.0;
        if (i < p) {
            const int col = SI(W.ix, i);
            const double* d = Dt + col * m;
            double a0 = 0.0, a1 = 0.0;
            int e = 0;
#pragma unroll 1
            for (; e + 1 < m; e += 2) {
                a0 = fma(__ldg(d + e), S[oR + e], a0);
                a1 = fma(__ldg(d + e + 1), S[oR + e + 1], a1);
            }
            if (e < m) a0 = fma(__ldg(d + e), S[oR + e], a0);
            double kx = 0.0;
#pragma unroll
            for (int dd = 0; dd < 5; ++dd) {
                const int c2 = col + dd - 2;
                if (c2 >= 0 && c2 < n) kx = fma(S[oKb + dd * n + col], S[W.xc + c2], kx);
            }
            gv[t] = (a0 + a1) - kx + S[oCp + col];
        }
    }
#pragma unroll
    for (int t = 0; t < NS; ++t) {
        const int i = lane + 32 * t;
        if (i < p) S[W.gs + i] = gv[t];
    }
    __syncwarp();
    double y[NS], dz[NS];
    tmul_transposed<NS>(W.T, W.gs, p, lane, y);
#pragma unroll
    for (int t = 0; t < NS; ++t) {
        const int i = lane + 32 * t;
        if (i < p) S[W.rs + i] = y[t];
    }
    __syncwarp();
    tmul<NS>(W.T, W.rs, p, lane, dz);
    bool ok = true;
#pragma unroll
    for (int t = 0; t < NS; ++t) {
        const int i = lane + 32 * t;
        if (i < p && !(S[W.xs + i] + dz[t] > 0.0)) ok = false;
    }
    if (__all_sync(FULL_MASK, ok)) {
#pragma unroll
        for (int t = 0; t < NS; ++t) {
            const int i = lane + 32 * t;
            if (i < p) {
                const double xn = S[W.xs + i] + dz[t];
                S[W.xs + i] = xn;
                S[W.xc + SI(W.ix, i)] = xn;
            }
        }
    }
    __syncwarp();
}

template <int NS, int ME>
__global__ void __launch_bounds__(SP_MAX_WARPS * 32) spatial_sweep_kernel(SpArgs A) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long it = (long long)blockIdx.x * (blockDim.x >> 5) + warp;
    if (it >= A.Vc) return;   // whole warps only
    const int n = A.n, m = A.m;
    const int base = warp * sp_warp_doubles<NS>(n);
    Slots<NS> W;
    W.carve(base, n);
    const int oM = base + Slots<NS>::doubles(n);
    const int oKb = oM + 64, oCp = oKb + 5 * n;
    const long long v = A.vox[it];
    if (v < 0 || v >= A.V) return;
    const int fa = A.fa_index[v];
    if ((A.status[v] & MET2_ST_SKIPPED) || fa < 0 || fa >= A.nA) return;   // not in the fitted set: x stays
    // y = sig / sig[0]
    const double km = A.sig[v * m];
#pragma unroll
    for (int u = 0; u < ME; ++u) {
        const int e = lane + 32 * u;
        if (e < m) S[oM + e] = A.sig[v * m + e] / km;
    }
    __syncwarp();
    // neighbours: n_v and the mean p of their rows (columns NS*lane + s, the layout of nnls_gram's column space)
    const int32_t* nb = A.nbr + v * 6;
    double ps[NS];
#pragma unroll
    for (int s = 0; s < NS; ++s) ps[s] = 0.0;
    int nv = 0;
    for (int f = 0; f < 6; ++f) {
        const long long q = nb[f];
        if (q < 0 || q >= A.V) continue;
        ++nv;
        const double* xq = A.x + q * n;
#pragma unroll
        for (int s = 0; s < NS; ++s) {
            const int col = NS * lane + s;
            if (col < n) ps[s] += xq[col];
        }
    }
    const double lamv = A.lam[v];
    const double w = A.mu * (double)nv;   // mu n_v
    const double* Dt = A.dicT + (size_t)fa * n * m;
    // c = D^T y + mu n_v p (lane owns columns NS*lane + s), the band lambda_v K + mu n_v I, the warm start (the
    // current support in column order: positions from a prefix count over the lanes)
    int cnt = 0;
#pragma unroll
    for (int s = 0; s < NS; ++s) {
        const int col = NS * lane + s;
        if (col < n) {
            const double* d = Dt + col * m;
            double a0 = 0.0, a1 = 0.0;
            int e = 0;
#pragma unroll 1
            for (; e + 1 < m; e += 2) {
                a0 = fma(__ldg(d + e), S[oM + e], a0);
                a1 = fma(__ldg(d + e + 1), S[oM + e + 1], a1);
            }
            if (e < m) a0 = fma(__ldg(d + e), S[oM + e], a0);
            const double cp = (nv > 0) ? w * (ps[s] / (double)nv) : 0.0;
            S[oCp + col] = cp;
            S[W.cc + col] = (a0 + a1) + cp;
#pragma unroll
            for (int d5 = 0; d5 < 5; ++d5) {
                double b = lamv * A.kband[d5 * n + col];
                if (d5 == 2) b += w;
                S[oKb + d5 * n + col] = b;
            }
            if (A.x[v * n + col] > 0.0) ++cnt;
        }
    }
    int pre = cnt;   // inclusive prefix over lanes
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(FULL_MASK, pre, o);
        if (lane >= o) pre += t;
    }
    const int p0 = __shfl_sync(FULL_MASK, pre, 31);
    int pos = pre - cnt;
#pragma unroll
    for (int s = 0; s < NS; ++s) {
        const int col = NS * lane + s;
        if (col < n) {
            const double xv = A.x[v * n + col];
            if (xv > 0.0) {
                SI(W.ix, pos) = col;
                S[W.xs + pos] = xv;
                ++pos;
            }
        }
    }
    set_dspace<NS>(W, nullptr, 0, lane);   // syncs the warp
    const double* Gg = A.G + (size_t)fa * n * n;
    int nst = 0;
    const int p = nnls_gram<NS, false, NS>(W, 0, Gg, n, oKb, true, 1.0, n, m + n, lane, nst, p0);
    if (nst == 0 && p > 0) refine_prior<NS, ME>(W, Dt, oM, m, p, lane, oKb, oCp, n);
#pragma unroll
    for (int s = 0; s < NS; ++s) {
        const int col = NS * lane + s;
        if (col < n) A.x[v * n + col] = S[W.xc + col];
    }
    if (nst && lane == 0) A.status[v] |= MET2_ST_ITMAX;
}

// fsol / est_signal / maps of the current x for every voxel: the output epilogue of met2_t2_impl.cuh
template <int NS, int ME>
__global__ void __launch_bounds__(SP_MAX_WARPS * 32)
    spatial_finish_kernel(const double* __restrict__ sig, const int32_t* __restrict__ fa_index,
                          const uint32_t* __restrict__ status, const double* __restrict__ x, long long V, int m, int n,
                          int nA, const double* __restrict__ dicT, const double* __restrict__ logT2,
                          const uint8_t* __restrict__ comp, double* __restrict__ fsol, double* __restrict__ est,
                          double* __restrict__ maps) {
    const int lane = threadIdx.x & 31;
    const long long v = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (v >= V) return;
    const int fa = fa_index[v];
    const bool fitted = !(status[v] & MET2_ST_SKIPPED) && fa >= 0 && fa < nA;
    const double kmo = fitted ? sig[v * m] : 0.0;
    double fit[ME];
#pragma unroll
    for (int u = 0; u < ME; ++u) fit[u] = 0.0;
    if (fitted) {
        const double* Dt = dicT + (size_t)fa * n * m;
        for (int j = 0; j < n; ++j) {
            const double xj = x[v * n + j];
            if (xj > 0.0) {
#pragma unroll
                for (int u = 0; u < ME; ++u) {
                    const int e = lane + 32 * u;
                    if (e < m) fit[u] = fma(__ldg(Dt + j * m + e), xj, fit[u]);
                }
            }
        }
    }
    double xk[NS];
    double vt = 0.0;
#pragma unroll
    for (int s = 0; s < NS; ++s) {
        const int col = NS * lane + s;
        xk[s] = (col < n && fitted) ? x[v * n + col] * kmo : 0.0;
        vt += xk[s];
        if (col < n) fsol[v * n + col] = xk[s];
    }
#pragma unroll
    for (int u = 0; u < ME; ++u) {
        const int e = lane + 32 * u;
        if (e < m) est[v * m + e] = fitted ? fit[u] * kmo : 0.0;
    }
    vt = warp_sum(vt) + 1.0e-16;
    double sm = 0.0, stt = 0.0, sc = 0.0, lm = 0.0, lt = 0.0;
#pragma unroll
    for (int s = 0; s < NS; ++s) {
        const int col = NS * lane + s;
        if (col < n) {
            const double xn = xk[s] / vt;
            const unsigned char cm = comp[col];
            if (cm & 1) {
                sm += xn;
                lm += xn * logT2[col];
            }
            if (cm & 2) {
                stt += xn;
                lt += xn * logT2[col];
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
        double* mp = maps + v * 6;
        mp[0] = sm;
        mp[1] = stt;
        mp[2] = sc;
        mp[3] = exp(lm / (sm + 1.0e-16));
        mp[4] = exp(lt / (stt + 1.0e-16));
        mp[5] = vt;
    }
}

static int sp_check_sizes(const char* what, int64_t V, int nTE, int nT2, int nA) {
    if (V < 0 || V > 0x7fffffffLL || nTE < 1 || nTE > MET2_MAX_NTE || nT2 < 1 || nT2 > MET2_MAX_NT2 || nA < 1)
        return set_error(MET2_ERR_ARG, "%s: bad sizes V=%lld nTE=%d nT2=%d nA=%d", what, (long long)V, nTE, nT2, nA);
    return MET2_OK;
}

template <int NS, int ME>
static int sp_launch_sweep(const SpArgs& A, cudaStream_t st) {
    const size_t per_warp = sizeof(double) * (size_t)sp_warp_doubles<NS>(A.n);
    int warps = (int)((227 * 1024 - 1024) / per_warp);
    if (warps > SP_MAX_WARPS) warps = SP_MAX_WARPS;
    const size_t smem = per_warp * warps;
    cudaError_t e = cudaFuncSetAttribute(spatial_sweep_kernel<NS, ME>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)smem);
    if (e != cudaSuccess) return set_error(MET2_ERR_CUDA, "spatial_sweep attr (%zu B): %s", smem, cudaGetErrorString(e));
    const long long blocks = (A.Vc + warps - 1) / warps;
    MET2_LAUNCH((unsigned)blocks, warps * 32, smem, st, spatial_sweep_kernel<NS, ME>)(A);
    count_launch();
    return check_launch("spatial_sweep_kernel");
}

}  // namespace met2

using namespace met2;

extern "C" int met2_spatial_sweep(const double* sig, const int32_t* fa_index, const double* lam, const int32_t* nbr,
                                  const int32_t* vox, int64_t Vc, int64_t V, int nTE, int nT2, int nA, const double* G,
                                  const double* dicT, const double* kband, double mu, double* x, uint32_t* status,
                                  void* stream) {
    int rc = sp_check_sizes("met2_spatial_sweep", V, nTE, nT2, nA);
    if (rc) return rc;
    if (Vc < 0 || Vc > V || !(mu >= 0.0) || !isfinite(mu))
        return set_error(MET2_ERR_ARG, "met2_spatial_sweep: bad argument (Vc=%lld, mu=%g)", (long long)Vc, mu);
    if (Vc > 0 && (!sig || !fa_index || !lam || !nbr || !vox || !G || !dicT || !kband || !x || !status))
        return set_error(MET2_ERR_ARG, "met2_spatial_sweep: NULL argument");
    if (Vc == 0) return MET2_OK;
    SpArgs A;
    A.sig = sig; A.fa_index = fa_index; A.lam = lam; A.nbr = nbr; A.vox = vox;
    A.V = V; A.Vc = Vc; A.m = nTE; A.n = nT2; A.nA = nA;
    A.G = G; A.dicT = dicT; A.kband = kband; A.mu = mu; A.x = x; A.status = status;
    cudaStream_t st = (cudaStream_t)stream;
    const int ns = (nT2 + 31) / 32, me = (nTE + 31) / 32;
    if (ns <= 2) return me == 1 ? sp_launch_sweep<2, 1>(A, st) : sp_launch_sweep<2, 2>(A, st);
    if (ns == 3) return me == 1 ? sp_launch_sweep<3, 1>(A, st) : sp_launch_sweep<3, 2>(A, st);
    return me == 1 ? sp_launch_sweep<4, 1>(A, st) : sp_launch_sweep<4, 2>(A, st);
}

extern "C" int met2_spatial_finish(const double* sig, const int32_t* fa_index, const uint32_t* status, const double* x,
                                   int64_t V, int nTE, int nT2, int nA, const double* dicT, const double* logT2,
                                   const uint8_t* comp, double* fsol, double* est_signal, double* maps, void* stream) {
    int rc = sp_check_sizes("met2_spatial_finish", V, nTE, nT2, nA);
    if (rc) return rc;
    if (V > 0 && (!sig || !fa_index || !status || !x || !dicT || !logT2 || !comp || !fsol || !est_signal || !maps))
        return set_error(MET2_ERR_ARG, "met2_spatial_finish: NULL argument");
    if (V == 0) return MET2_OK;
    cudaStream_t st = (cudaStream_t)stream;
    const unsigned blocks = (unsigned)((V + SP_MAX_WARPS - 1) / SP_MAX_WARPS);
    const int ns = (nT2 + 31) / 32, me = (nTE + 31) / 32;
#define SP_FINISH(NS_, ME_)                                                                                          \
    MET2_LAUNCH(blocks, SP_MAX_WARPS * 32, 0, st, spatial_finish_kernel<NS_, ME_>)(                                  \
        sig, fa_index, status, x, (long long)V, nTE, nT2, nA, dicT, logT2, comp, fsol, est_signal, maps)
    if (ns <= 2) {
        if (me == 1) SP_FINISH(2, 1); else SP_FINISH(2, 2);
    } else if (ns == 3) {
        if (me == 1) SP_FINISH(3, 1); else SP_FINISH(3, 2);
    } else {
        if (me == 1) SP_FINISH(4, 1); else SP_FINISH(4, 2);
    }
#undef SP_FINISH
    count_launch();
    return check_launch("met2_spatial_finish");
}
