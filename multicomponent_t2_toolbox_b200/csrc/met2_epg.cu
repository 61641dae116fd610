// met2_epg.cu — EPG dictionary, Gram tables and band forms (run once per reconstruction).
//
// Takes over epg/epg.py:155 create_Dic_3D -> :47 create_met2_design_matrix_epg -> :64 epg_signal.  The reference builds
// dense (3n+1)^2 matrices S (shift), R (relaxation over tau/2), T (RF) and iterates x <- (R S) T (R S) x per echo
// (epg.py:89-91,143-153).  Here one thread owns one (flip angle, T2) pair and applies the same operator sequence
// directly to the banded state (F0; F+k, F-k, Zk, k = 1..n): shift, relax, RF, shift, relax; O(n^2) instead of O(n^3).
// The coefficients and block operators are those of met2_epg.cuh, shared with the parametric fit (met2_param.cu).
#include "met2_host.h"
#include "met2_epg.cuh"

#ifdef MET2_HOST_EMU
#define __grid_constant__
#endif

namespace met2 {

__device__ __forceinline__ void epg_train(const EpgCoef<double>& c, int n, double scale, double* out, int out_stride) {
    double Fp[MET2_MAX_NTE + 2], Fm[MET2_MAX_NTE + 2], Z[MET2_MAX_NTE + 2];
    for (int k = 0; k < n + 2; ++k) Fp[k] = Fm[k] = Z[k] = 0.0;
    double F0 = c.f0;
    Fm[1] = c.fm1;
    for (int echo = 0; echo < n; ++echo) {
        for (int half_step = 0; half_step < 2; ++half_step) {
            // shift (epg.py:97-116): F0 <- F-1, F+1 <- F0, F+k <- F+(k-1), F-k <- F-(k+1), F-n <- 0
            double newF0 = Fm[1];
            for (int k = n; k >= 2; --k) Fp[k] = Fp[k - 1];
            Fp[1] = F0;
            for (int k = 1; k < n; ++k) Fm[k] = Fm[k + 1];
            Fm[n] = 0.0;
            F0 = newF0 * c.e2;
            for (int k = 1; k <= n; ++k) epg_relax(Fp[k], Fm[k], Z[k], c);
            if (half_step == 0)
                for (int k = 1; k <= n; ++k) epg_rf(Fp[k], Fm[k], Z[k], c);
        }
        out[(size_t)echo * out_stride] = scale * F0;
    }
}

__device__ __forceinline__ void epg_decay(double alpha_deg, double T2, double T1, int n, double tau, double scale,
                                          double* out, int out_stride) {
    epg_train(epg_coef(alpha_deg, T2, T1, tau), n, scale, out, out_stride);
}

__global__ void epg_dictionary_kernel(const double* __restrict__ alphas, int nA, const double* __restrict__ T2s,
                                      const double* __restrict__ T1s, int nT2, int nTE, double tau, double TR,
                                      double* __restrict__ dic, double* __restrict__ dicT) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nA * nT2) return;
    int a = i / nT2, j = i - a * nT2;
    double tmp[MET2_MAX_NTE];
    double scale = 1.0 - exp(-TR / T1s[j]);   // epg.py:57
    epg_decay(alphas[a], T2s[j], T1s[j], nTE, tau, scale, tmp, 1);
    for (int e = 0; e < nTE; ++e) {
        if (dic) dic[((size_t)a * nTE + e) * nT2 + j] = tmp[e];
        if (dicT) dicT[((size_t)a * nT2 + j) * nTE + e] = tmp[e];
    }
}

__global__ void epg_signals_kernel(const double* __restrict__ alphas, const double* __restrict__ T2s,
                                   const double* __restrict__ T1s, long long N, int nTE, double tau,
                                   double* __restrict__ sig) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    epg_decay(alphas[i], T2s[i], T1s[i], nTE, tau, 1.0, sig + i * nTE, 1);
}

// ---------------------------------------------------------------------------------------------------- slice profile
// Profile-integrated echo trains for 2-D multi-slice CPMG (DESIGN §10g).  A slice profile is K positions with
// excitation scale x[k], refocusing scale r[k] and weight w[k]; at nominal angle alpha the curve is
//     S_e = sum_{k = 0..K-1, in this order}  w[k] * EPG_e(T2, T1, refocusing = alpha r[k], excitation = (alpha/2) x[k])
// with EPG_e the recurrence above (epg_train).  One block per curve: the threads run the K trains C = blockDim.x at a
// time into sT[e][C] (shared), then the owner of echo e (thread e mod C) adds the chunk's C terms to sA[e] one after the
// other.  The sum order is therefore k = 0, 1, ..., K-1 whatever the block size or the scheduling of the threads, and
// K = 1 with x = r = w = 1 gives 0 + 1 * F0 = the train of epg_decay bit for bit.
// The profile is passed by value (12 KB of kernel parameters): it is checked on the host before any launch.
struct ProfileTab {
    double x[MET2_MAX_PROFILE], r[MET2_MAX_PROFILE], w[MET2_MAX_PROFILE];
};

__device__ __forceinline__ void profile_train(double alpha, double T2, double T1, int nTE, double tau,
                                              const ProfileTab& p, int K, double* sT, double* sA) {
    const int C = blockDim.x, t = threadIdx.x;
    for (int e = t; e < nTE; e += C) sA[e] = 0.0;
    for (int k0 = 0; k0 < K; k0 += C) {
        const int k = k0 + t;
        if (k < K) epg_train(epg_coef(alpha * p.r[k], (alpha / 2.0) * p.x[k], T2, T1, tau), nTE, 1.0, sT + t, C);
        __syncthreads();
        const int cnt = min(C, K - k0);
        for (int e = t; e < nTE; e += C) {
            double s = sA[e];
            for (int i = 0; i < cnt; ++i) s = s + p.w[k0 + i] * sT[e * C + i];
            sA[e] = s;
        }
        __syncthreads();
    }
}

__global__ void epg_dictionary_profile_kernel(const double* __restrict__ alphas, const double* __restrict__ T2s,
                                              const double* __restrict__ T1s, int nT2, int nTE, double tau, double TR,
                                              const __grid_constant__ ProfileTab p, int K, double* __restrict__ dic,
                                              double* __restrict__ dicT) {
#ifdef MET2_HOST_EMU
    double* sT = simt::g_shared.data;
#else
    extern __shared__ double sT[];
#endif
    double* sA = sT + (size_t)nTE * blockDim.x;
    const int a = blockIdx.x / nT2, j = blockIdx.x - a * nT2;
    profile_train(alphas[a], T2s[j], T1s[j], nTE, tau, p, K, sT, sA);
    const double scale = 1.0 - exp(-TR / T1s[j]);   // epg.py:57
    for (int e = threadIdx.x; e < nTE; e += blockDim.x) {
        const double v = scale * sA[e];
        if (dic) dic[((size_t)a * nTE + e) * nT2 + j] = v;
        if (dicT) dicT[((size_t)a * nT2 + j) * nTE + e] = v;
    }
}

__global__ void epg_signals_profile_kernel(const double* __restrict__ alphas, const double* __restrict__ T2s,
                                           const double* __restrict__ T1s, int nTE, double tau,
                                           const __grid_constant__ ProfileTab p, int K, double* __restrict__ sig) {
#ifdef MET2_HOST_EMU
    double* sT = simt::g_shared.data;
#else
    extern __shared__ double sT[];
#endif
    double* sA = sT + (size_t)nTE * blockDim.x;
    const size_t i = blockIdx.x;
    profile_train(alphas[i], T2s[i], T1s[i], nTE, tau, p, K, sT, sA);
    for (int e = threadIdx.x; e < nTE; e += blockDim.x) sig[i * nTE + e] = sA[e];
}

// G[a] = D_a^T D_a, one block per angle; D_a staged in shared memory.
__global__ void gram_kernel(const double* __restrict__ dic, int nTE, int nT2, double* __restrict__ G) {
#ifdef MET2_HOST_EMU
    double* sD = simt::g_shared.data;
#else
    extern __shared__ double sD[];
#endif
    const double* D = dic + (size_t)blockIdx.x * nTE * nT2;
    for (int i = threadIdx.x; i < nTE * nT2; i += blockDim.x) sD[i] = D[i];
    __syncthreads();
    double* Ga = G + (size_t)blockIdx.x * nT2 * nT2;
    for (int ij = threadIdx.x; ij < nT2 * nT2; ij += blockDim.x) {
        int i = ij / nT2, j = ij - i * nT2;
        double acc = 0.0;
        for (int e = 0; e < nTE; ++e) acc = fma(sD[e * nT2 + i], sD[e * nT2 + j], acc);
        Ga[ij] = acc;
    }
}

// kband rows 0..4: K = L^T L in column band form kb[d][c] = K[c+d-2][c]; rows 5..9: L in row band form
// lb[d][r] = L[r][r+d-2].  band_err := 1 if K or L has a non-zero outside the five central diagonals.
__global__ void band_kernel(const double* __restrict__ L, int n, double* __restrict__ kband, int* __restrict__ band_err) {
    for (int rc = threadIdx.x; rc < n * n; rc += blockDim.x) {
        int r = rc / n, c = rc - r * n;
        double k = 0.0;
        for (int i = 0; i < n; ++i) k = fma(L[i * n + r], L[i * n + c], k);
        int d = r - c + 2;
        if (d >= 0 && d <= 4) {
            kband[d * n + c] = k;
        } else if (k != 0.0 && band_err) {
            *band_err = 1;
        }
        int dl = c - r + 2;
        if (dl >= 0 && dl <= 4) {
            kband[(5 + dl) * n + r] = L[r * n + c];
        } else if (L[r * n + c] != 0.0 && band_err) {
            *band_err = 1;
        }
    }
}


}  // namespace met2

using namespace met2;

extern "C" int met2_epg_dictionary(const double* alphas_deg, int nA, const double* T2s, const double* T1s, int nT2,
                                   int nTE, double tau_ms, double TR_ms, double* dic, double* dicT, void* stream) {
    if (!alphas_deg || !T2s || !T1s || nA <= 0 || nT2 <= 0 || nT2 > MET2_MAX_NT2 || nTE <= 0 || nTE > MET2_MAX_NTE)
        return set_error(MET2_ERR_ARG, "met2_epg_dictionary: bad argument (nA=%d nT2=%d nTE=%d)", nA, nT2, nTE);
    cudaStream_t st = (cudaStream_t)stream;
    int total = nA * nT2;
    MET2_LAUNCH((total + 127) / 128, 128, 0, st, epg_dictionary_kernel)(alphas_deg, nA, T2s, T1s, nT2, nTE, tau_ms, TR_ms, dic,
                                                               dicT);
    count_launch();
    return check_launch("epg_dictionary_kernel");
}

extern "C" int met2_epg_signals(const double* alphas_deg, const double* T2s, const double* T1s, int64_t N, int nTE,
                                double tau_ms, double* sig, void* stream) {
    if (!alphas_deg || !T2s || !T1s || !sig || N < 0 || nTE <= 0 || nTE > MET2_MAX_NTE)
        return set_error(MET2_ERR_ARG, "met2_epg_signals: bad argument");
    if (N == 0) return MET2_OK;
    cudaStream_t st = (cudaStream_t)stream;
    MET2_LAUNCH((unsigned)((N + 127) / 128), 128, 0, st, epg_signals_kernel)(alphas_deg, T2s, T1s, (long long)N, nTE, tau_ms, sig);
    count_launch();
    return check_launch("epg_signals_kernel");
}

namespace {

// K in 1..MET2_MAX_PROFILE and every x / r / w finite and >= 0 (host arrays) -> the kernels' table; else MET2_ERR_ARG.
int profile_table(const char* what, const double* x, const double* r, const double* w, int K, ProfileTab* p) {
    if (!x || !r || !w || K < 1 || K > MET2_MAX_PROFILE)
        return set_error(MET2_ERR_ARG, "%s: bad slice profile (K=%d, 1..%d positions)", what, K, MET2_MAX_PROFILE);
    for (int k = 0; k < K; ++k) {
        const double v[3] = {x[k], r[k], w[k]};
        for (double q : v)
            if (!(q >= 0.0 && q <= 1.7976931348623157e308))   // false for NaN, negatives and +Inf
                return set_error(MET2_ERR_ARG, "%s: slice profile entry %d is not finite and >= 0", what, k);
        p->x[k] = x[k];
        p->r[k] = r[k];
        p->w[k] = w[k];
    }
    return MET2_OK;
}

// 32 threads for up to 32 positions, else 64 (one chunk of trains at the K = 64 of the default profile)
int profile_threads(int K) { return K <= 32 ? 32 : 64; }

}  // namespace

extern "C" int met2_epg_dictionary_profile(const double* alphas_deg, int nA, const double* T2s, const double* T1s,
                                           int nT2, int nTE, double tau_ms, double TR_ms, const double* x,
                                           const double* r, const double* w, int K, double* dic, double* dicT,
                                           void* stream) {
    if (!alphas_deg || !T2s || !T1s || nA <= 0 || nT2 <= 0 || nT2 > MET2_MAX_NT2 || nTE <= 0 || nTE > MET2_MAX_NTE ||
        (int64_t)nA * nT2 > INT32_MAX)
        return set_error(MET2_ERR_ARG, "met2_epg_dictionary_profile: bad argument (nA=%d nT2=%d nTE=%d)", nA, nT2, nTE);
    ProfileTab p;
    int rc = profile_table("met2_epg_dictionary_profile", x, r, w, K, &p);
    if (rc) return rc;
    const int C = profile_threads(K);
    MET2_LAUNCH(nA * nT2, C, sizeof(double) * (size_t)nTE * (C + 1), (cudaStream_t)stream,
                epg_dictionary_profile_kernel)(alphas_deg, T2s, T1s, nT2, nTE, tau_ms, TR_ms, p, K, dic, dicT);
    count_launch();
    return check_launch("epg_dictionary_profile_kernel");
}

extern "C" int met2_epg_signals_profile(const double* alphas_deg, const double* T2s, const double* T1s, int64_t N,
                                        int nTE, double tau_ms, const double* x, const double* r, const double* w,
                                        int K, double* sig, void* stream) {
    if (!alphas_deg || !T2s || !T1s || !sig || N < 0 || N > INT32_MAX || nTE <= 0 || nTE > MET2_MAX_NTE)
        return set_error(MET2_ERR_ARG, "met2_epg_signals_profile: bad argument");
    ProfileTab p;
    int rc = profile_table("met2_epg_signals_profile", x, r, w, K, &p);
    if (rc) return rc;
    if (N == 0) return MET2_OK;
    const int C = profile_threads(K);
    MET2_LAUNCH((unsigned)N, C, sizeof(double) * (size_t)nTE * (C + 1), (cudaStream_t)stream,
                epg_signals_profile_kernel)(alphas_deg, T2s, T1s, nTE, tau_ms, p, K, sig);
    count_launch();
    return check_launch("epg_signals_profile_kernel");
}

extern "C" int met2_gram_tables(const double* dic, int nA, int nTE, int nT2, const double* L, double* G, double* kband,
                                int32_t* band_err, void* stream) {
    if (nA < 0 || nT2 <= 0 || nT2 > MET2_MAX_NT2 || nTE <= 0 || nTE > MET2_MAX_NTE)
        return set_error(MET2_ERR_ARG, "met2_gram_tables: bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    if (dic && G && nA > 0) {
        size_t smem = sizeof(double) * (size_t)nTE * nT2;
        cudaError_t e = cudaFuncSetAttribute(gram_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return set_error(MET2_ERR_CUDA, "gram_kernel attr: %s", cudaGetErrorString(e));
        MET2_LAUNCH(nA, 256, smem, st, gram_kernel)(dic, nTE, nT2, G);
        count_launch();
        int rc = check_launch("gram_kernel");
        if (rc) return rc;
    }
    if (L && kband) {
        cudaError_t e = cudaMemsetAsync(kband, 0, sizeof(double) * 10 * nT2, st);
        if (e != cudaSuccess) return set_error(MET2_ERR_CUDA, "memset kband: %s", cudaGetErrorString(e));
        if (band_err) cudaMemsetAsync(band_err, 0, sizeof(int32_t), st);
        MET2_LAUNCH(1, 256, 0, st, band_kernel)(L, nT2, kband, band_err);
        count_launch();
        return check_launch("band_kernel");
    }
    return MET2_OK;
}
