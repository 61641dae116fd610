// met2_rician.cu — Rician-likelihood spectrum fitting (no counterpart in the reference): majorize-minimize (MM)
// iterations of warm-started Tikhonov NNLS solves with modified data (Varadarajan & Haldar, IEEE TMI 2015), started
// from the point fit (met2_t2_fit).  Nothing here selects lambda.
//
// Definition (tests/rician_oracle.py restates it in NumPy; DESIGN.md §10f).  All quantities are in the reference's
// normalised units.  For a fitted voxel v of the point fit (status without MET2_ST_SKIPPED):
//   y = sig_v / sig_v[0],  x^0 = x0_v (fsol_v / sig_v[0]),  a = fa_index[v],  lambda = lam[v] (any lam[v] >= 0; the
//   pipeline passes the point fit's lambda, reg under MET2_T2_FLAG_REG_IS_LAMBDA),  sn = sigma[v] / sig_v[0] with
//   sigma the noise SD in raw signal units,  s2 = sn * sn.
// Objective, f = D_a x, x >= 0:
//   Phi(x) = sum_e [ f_e^2 - 2 s2 log I0(y_e f_e / s2) ] + lambda ||L x||^2,
//   2 s2 times the Rician negative log-likelihood plus the Tikhonov term; it tends to ||D x - y||^2 + lambda ||L x||^2
//   as sn -> 0.
// MM step: log I0 is convex, so -2 s2 log I0 is majorised by its tangent line, which gives
//   yt_e = y_e * A((y_e * f_e) / s2),  A = I1 / I0,   x <- argmin_{x >= 0} ||D_a x - yt||^2 + lambda ||L x||^2,
//   and Phi never increases.
// A(z) (rc_bessel_ratio): Cephes' i0e / i1e Chebyshev tables (the ones SciPy and ATen carry); the exp and sqrt factors
// cancel in the ratio:  z <= 8: A = (z * chbevl(z/2 - 2, A1, 29)) / chbevl(z/2 - 2, A0, 30);  z > 8: A =
// chbevl(32/z - 2, B1, 25) / chbevl(32/z - 2, B0, 25);  A(-z) = -A(z).  Only IEEE +, -, *, / (the library is built
// with -fmad=false), one __host__ __device__ routine: met2_bessel_ratio runs the same code on the host, and NumPy
// reproduces it bit for bit.  z = +inf gives 32/inf - 2 = -2 and exactly 1.0.
// Loop: yt^0 = y.  For k = 1 .. max_iter:  f = D_a x^{k-1};  form yt^k;  if max_e |yt^k_e - yt^{k-1}_e| <= tol stop
//   with iters = k - 1;  else x^k = the solve with yt^k, warm-started from x^{k-1}'s support and coefficients.  A loop
//   that runs max_iter solves ends with iters = max_iter and MET2_ST_MM_CAP.
// Special cases: s2 = 0 (sigma = 0) gives yt = y without evaluating A (0/0 is possible), so the voxel stops at
//   iters = 0 with x = x^0: the point fit.  A NaN, +-Inf or negative sigma[v] gives x = 0 and MET2_ST_BAD_SIGMA |
//   MET2_ST_SKIPPED.  A solve that hits itmax ORs MET2_ST_ITMAX.  Voxels the point fit skipped get x = 0, iters = 0 and
//   their status unchanged.
// Outputs: x [V][nT2], iters [V] int32, status [V] (the point fit's plus the bits above); met2_spatial_finish then gives
//   fsol = x sig[0], est_signal = D_a x sig[0] (the noiseless model, not the Rician mean) and the six maps.
//
// met2_rician_fit: one warp per voxel, RC_MAX_WARPS warps per block and no block-wide barrier (as met2_spatial_sweep).
// Per-warp shared memory holds the NNLS slots, y, yt (in the signal slot the solver and refine_on_support read) and the
// 5-band lambda K.  Each solve is the Gram-domain Lawson-Hanson of met2_nnls.cuh with c = D^T yt, warm-started from the
// previous support (the first from x^0's support in column order), with the D-space candidate test on for the plain
// problem (as the point fit's NNLS) and the D-space refinement step of met2_device.cuh on the final support.  The
// minimiser of each (convex) surrogate problem does not depend on the start.
#include <math.h>

#include "met2_device.cuh"
#include "met2_host.h"

namespace met2 {

constexpr int RC_MAX_WARPS = 4;   // voxels per block (no block-wide barrier: warps retire independently)

// Clenshaw sum of Cephes' chbevl: b0 = c[0]; b0 <- x b1 - b2 + c[k] for k = 1 .. n-1; 0.5 (b0 - b2)
template <int N>
__host__ __device__ inline double rc_chbevl(double x, const double (&c)[N]) {
    double b0 = c[0], b1 = 0.0, b2 = 0.0;
#pragma unroll
    for (int k = 1; k < N; ++k) {
        b2 = b1;
        b1 = b0;
        b0 = x * b1 - b2 + c[k];
    }
    return 0.5 * (b0 - b2);
}

// A(z) = I1(z) / I0(z) (see the header)
__host__ __device__ inline double rc_bessel_ratio(double z) {
    const double A0[30] = {
        -4.41534164647933937950E-18, 3.33079451882223809783E-17, -2.43127984654795469359E-16,
        1.71539128555513303061E-15, -1.16853328779934516808E-14, 7.67618549860493561688E-14,
        -4.85644678311192946090E-13, 2.95505266312963983461E-12, -1.72682629144155570723E-11,
        9.67580903537323691224E-11, -5.18979560163526290666E-10, 2.65982372468238665035E-9,
        -1.30002500998624804212E-8, 6.04699502254191894932E-8, -2.67079385394061173391E-7,
        1.11738753912010371815E-6, -4.41673835845875056359E-6, 1.64484480707288970893E-5,
        -5.75419501008210370398E-5, 1.88502885095841655729E-4, -5.76375574538582365885E-4,
        1.63947561694133579842E-3, -4.32430999505057594430E-3, 1.05464603945949983183E-2,
        -2.37374148058994688156E-2, 4.93052842396707084878E-2, -9.49010970480476444210E-2,
        1.71620901522208775349E-1, -3.04682672343198398683E-1, 6.76795274409476084995E-1};
    const double A1[29] = {
        2.77791411276104639959E-18, -2.11142121435816608115E-17, 1.55363195773620046921E-16,
        -1.10559694773538630805E-15, 7.60068429473540693410E-15, -5.04218550472791168711E-14,
        3.22379336594557470981E-13, -1.98397439776494371520E-12, 1.17361862988909016308E-11,
        -6.66348972350202774223E-11, 3.62559028155211703701E-10, -1.88724975172282928790E-9,
        9.38153738649577178388E-9, -4.44505912879632808065E-8, 2.00329475355213526229E-7,
        -8.56872026469545474066E-7, 3.47025130813767847674E-6, -1.32731636560394358279E-5,
        4.78156510755005422638E-5, -1.61760815825896745588E-4, 5.12285956168575772895E-4,
        -1.51357245063125314899E-3, 4.15642294431288815669E-3, -1.05640848946261981558E-2,
        2.47264490306265168283E-2, -5.29459812080949914269E-2, 1.02643658689847095384E-1,
        -1.76416518357834055153E-1, 2.52587186443633654823E-1};
    const double B0[25] = {
        -7.23318048787475395456E-18, -4.83050448594418207126E-18, 4.46562142029675999901E-17,
        3.46122286769746109310E-17, -2.82762398051658348494E-16, -3.42548561967721913462E-16,
        1.77256013305652638360E-15, 3.81168066935262242075E-15, -9.55484669882830764870E-15,
        -4.15056934728722208663E-14, 1.54008621752140982691E-14, 3.85277838274214270114E-13,
        7.18012445138366623367E-13, -1.79417853150680611778E-12, -1.32158118404477131188E-11,
        -3.14991652796324136454E-11, 1.18891471078464383424E-11, 4.94060238822496958910E-10,
        3.39623202570838634515E-9, 2.26666899049817806459E-8, 2.04891858946906374183E-7,
        2.89137052083475648297E-6, 6.88975834691682398426E-5, 3.36911647825569408990E-3,
        8.04490411014108831608E-1};
    const double B1[25] = {
        7.51729631084210481353E-18, 4.41434832307170791151E-18, -4.65030536848935832153E-17,
        -3.20952592199342395980E-17, 2.96262899764595013876E-16, 3.30820231092092828324E-16,
        -1.88035477551078244854E-15, -3.81440307243700780478E-15, 1.04202769841288027642E-14,
        4.27244001671195135429E-14, -2.10154184277266431302E-14, -4.08355111109219731823E-13,
        -7.19855177624590851209E-13, 2.03562854414708950722E-12, 1.41258074366137813316E-11,
        3.25260358301548823856E-11, -1.89749581235054123450E-11, -5.58974346219658380687E-10,
        -3.83538038596423702205E-9, -2.63146884688951950684E-8, -2.51223623787020892529E-7,
        -3.88256480887769039346E-6, -1.10588938762623716291E-4, -9.76109749136146840777E-3,
        7.78576235018280120474E-1};
    const double a = z < 0.0 ? -z : z;
    double r;
    if (a <= 8.0) {
        const double t = a / 2.0 - 2.0;
        r = (a * rc_chbevl(t, A1)) / rc_chbevl(t, A0);
    } else {
        const double t = 32.0 / a - 2.0;
        r = rc_chbevl(t, B1) / rc_chbevl(t, B0);
    }
    return z < 0.0 ? -r : r;
}

struct RcArgs {
    const double* sig;          // [V][m] raw signals
    const int32_t* fa_index;    // [V]
    const double* lam;          // [V] lambda_v
    const double* sigma;        // [V] noise SD, raw units
    const double* x0;           // [V][n] normalised point-fit spectra
    const uint32_t* status_in;  // [V]
    long long V;
    int m, n, nA, max_iter;
    double tol;
    const double *G, *dicT, *kband;
    double* x;                  // [V][n]
    int32_t* iters;             // [V]
    uint32_t* status;           // [V]
};

// per-warp shared memory: [NNLS slots (pmax = n)][yt 64][y 64][band 5n]
template <int NS>
__host__ __device__ __forceinline__ int rc_warp_doubles(int n) {
    return (Slots<NS>::doubles(n) + 128 + 5 * n + 31) & ~31;
}

template <int NS, int ME>
__global__ void __launch_bounds__(RC_MAX_WARPS * 32, 1) rician_kernel(RcArgs A) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long v = (long long)blockIdx.x * (blockDim.x >> 5) + warp;
    if (v >= A.V) return;   // whole warps only
    const int n = A.n, m = A.m;
    const int base = warp * rc_warp_doubles<NS>(n);
    Slots<NS> W;
    W.carve(base, n);
    const int oM = base + Slots<NS>::doubles(n);   // yt: the solver's right-hand side
    const int oY = oM + 64, oKb = oY + 64;
    unsigned st = A.status_in[v];
    const int fa = A.fa_index[v];
    const double sg = A.sigma[v];
    bool fitted = !(st & MET2_ST_SKIPPED) && fa >= 0 && fa < A.nA;
    if (fitted && !(isfinite(sg) && sg >= 0.0)) {
        st |= MET2_ST_BAD_SIGMA | MET2_ST_SKIPPED;
        fitted = false;
    }
    if (!fitted) {
#pragma unroll
        for (int s = 0; s < NS; ++s) {
            const int col = NS * lane + s;
            if (col < n) A.x[v * n + col] = 0.0;
        }
        if (lane == 0) {
            A.iters[v] = 0;
            A.status[v] = st;
        }
        return;
    }
    // y = sig / sig[0]; yt^0 = y
    const double km = A.sig[v * m];
#pragma unroll
    for (int u = 0; u < ME; ++u) {
        const int e = lane + 32 * u;
        if (e < m) {
            const double yv = A.sig[v * m + e] / km;
            S[oY + e] = yv;
            S[oM + e] = yv;
        }
    }
    const double sn = sg / km;
    const double s2 = sn * sn;
    const double lamv = A.lam[v];
    const bool reg = lamv > 0.0;
    const double* Dt = A.dicT + (size_t)fa * n * m;
    const double* Gg = A.G + (size_t)fa * n * n;
    // the band lambda K, x^0 in column space and its support in column order (positions from a prefix count)
    int cnt = 0;
#pragma unroll
    for (int s = 0; s < NS; ++s) {
        const int col = NS * lane + s;
        if (col < n) {
#pragma unroll
            for (int d5 = 0; d5 < 5; ++d5) S[oKb + d5 * n + col] = lamv * A.kband[d5 * n + col];
            const double xv = A.x0[v * n + col];
            S[W.xc + col] = xv > 0.0 ? xv : 0.0;
            if (xv > 0.0) ++cnt;
        }
    }
    int pre = cnt;   // inclusive prefix over lanes
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(FULL_MASK, pre, o);
        if (lane >= o) pre += t;
    }
    int p = __shfl_sync(FULL_MASK, pre, 31);
    int pos = pre - cnt;
#pragma unroll
    for (int s = 0; s < NS; ++s) {
        const int col = NS * lane + s;
        if (col < n) {
            const double xv = A.x0[v * n + col];
            if (xv > 0.0) {
                SI(W.ix, pos) = col;
                S[W.xs + pos] = xv;
                ++pos;
            }
        }
    }
    set_dspace<NS>(W, Dt, oM, lane);   // syncs the warp
    int iters = A.max_iter, nst = 0;
    bool capped = true;
    for (int k = 1; k <= A.max_iter; ++k) {
        double fit[ME];
        (void)fit_and_sse<NS, ME>(W, Dt, oM, m, p, lane, fit);   // f = D x^{k-1}
        double yt[ME], dmax = 0.0;
#pragma unroll
        for (int u = 0; u < ME; ++u) {
            const int e = lane + 32 * u;
            yt[u] = 0.0;
            if (e < m) {
                const double yv = S[oY + e];
                yt[u] = s2 > 0.0 ? yv * rc_bessel_ratio((yv * fit[u]) / s2) : yv;
                dmax = fmax(dmax, fabs(yt[u] - S[oM + e]));
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) dmax = fmax(dmax, __shfl_xor_sync(FULL_MASK, dmax, o));
        __syncwarp();
        if (dmax <= A.tol) {
            iters = k - 1;
            capped = false;
            break;
        }
#pragma unroll
        for (int u = 0; u < ME; ++u) {
            const int e = lane + 32 * u;
            if (e < m) S[oM + e] = yt[u];
        }
        __syncwarp();
        // c = D^T yt (lane owns columns NS*lane + s)
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
                S[W.cc + col] = a0 + a1;
            }
        }
        __syncwarp();
        int ns1 = 0;
        p = nnls_gram<NS, false, NS>(W, 0, Gg, n, oKb, reg, 1.0, n, reg ? m + n : m, lane, ns1, p);
        if (ns1 == 0 && p > 0) refine_on_support<NS, ME>(W, Dt, oM, m, p, lane, reg, 1.0, oKb, n);
        nst |= ns1;
    }
#pragma unroll
    for (int s = 0; s < NS; ++s) {
        const int col = NS * lane + s;
        if (col < n) A.x[v * n + col] = S[W.xc + col];
    }
    if (capped) st |= MET2_ST_MM_CAP;
    if (nst) st |= MET2_ST_ITMAX;
    if (lane == 0) {
        A.iters[v] = iters;
        A.status[v] = st;
    }
}

template <int NS, int ME>
static int rc_launch(const RcArgs& A, cudaStream_t st) {
    const size_t per_warp = sizeof(double) * (size_t)rc_warp_doubles<NS>(A.n);
    int warps = (int)((227 * 1024 - 1024) / per_warp);
    if (warps > RC_MAX_WARPS) warps = RC_MAX_WARPS;
    const size_t smem = per_warp * warps;
    cudaError_t e = cudaFuncSetAttribute(rician_kernel<NS, ME>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return set_error(MET2_ERR_CUDA, "rician attr (%zu B): %s", smem, cudaGetErrorString(e));
    const long long blocks = (A.V + warps - 1) / warps;
    MET2_LAUNCH((unsigned)blocks, warps * 32, smem, st, rician_kernel<NS, ME>)(A);
    count_launch();
    return check_launch("rician_kernel");
}

}  // namespace met2

using namespace met2;

extern "C" int met2_rician_fit(const double* sig, const int32_t* fa_index, const double* lam, const double* sigma,
                               const double* x0, const uint32_t* status_in, int64_t V, int nTE, int nT2, int nA,
                               const double* G, const double* dicT, const double* kband, int max_iter, double tol,
                               double* x, int32_t* iters, uint32_t* status, void* stream) {
    if (V < 0 || V > 0x7fffffffLL || nTE < 1 || nTE > MET2_MAX_NTE || nT2 < 1 || nT2 > MET2_MAX_NT2 || nA < 1)
        return set_error(MET2_ERR_ARG, "met2_rician_fit: bad sizes V=%lld nTE=%d nT2=%d nA=%d", (long long)V, nTE, nT2,
                         nA);
    if (max_iter < 1 || !(tol >= 0.0) || !isfinite(tol))
        return set_error(MET2_ERR_ARG, "met2_rician_fit: bad argument (max_iter=%d, tol=%g)", max_iter, tol);
    if (V > 0 && (!sig || !fa_index || !lam || !sigma || !x0 || !status_in || !G || !dicT || !kband || !x || !iters ||
                  !status))
        return set_error(MET2_ERR_ARG, "met2_rician_fit: NULL argument");
    if (V == 0) return MET2_OK;
    RcArgs A;
    A.sig = sig; A.fa_index = fa_index; A.lam = lam; A.sigma = sigma; A.x0 = x0; A.status_in = status_in;
    A.V = V; A.m = nTE; A.n = nT2; A.nA = nA; A.max_iter = max_iter; A.tol = tol;
    A.G = G; A.dicT = dicT; A.kband = kband; A.x = x; A.iters = iters; A.status = status;
    cudaStream_t st = (cudaStream_t)stream;
    const int ns = (nT2 + 31) / 32, me = (nTE + 31) / 32;
    if (ns <= 2) return me == 1 ? rc_launch<2, 1>(A, st) : rc_launch<2, 2>(A, st);
    if (ns == 3) return me == 1 ? rc_launch<3, 1>(A, st) : rc_launch<3, 2>(A, st);
    return me == 1 ? rc_launch<4, 1>(A, st) : rc_launch<4, 2>(A, st);
}

extern "C" int64_t met2_bessel_ratio(const double* z, int64_t n, double* out) {
    if (n < 0 || (n > 0 && (!z || !out)))
        return set_error(MET2_ERR_ARG, "met2_bessel_ratio: bad argument (n=%lld)", (long long)n);
    for (int64_t i = 0; i < n; ++i) out[i] = rc_bessel_ratio(z[i]);
    return n;
}
