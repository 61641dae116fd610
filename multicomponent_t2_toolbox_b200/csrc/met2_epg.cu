// met2_epg.cu — EPG dictionary, Gram tables and band forms (run once per reconstruction).
//
// Takes over epg/epg.py:155 create_Dic_3D -> :47 create_met2_design_matrix_epg -> :64 epg_signal.  The reference builds
// dense (3n+1)^2 matrices S (shift), R (relaxation over tau/2), T (RF) and iterates x <- (R S) T (R S) x per echo
// (epg.py:89-91,143-153).  Here one thread owns one (flip angle, T2) pair and applies the same operator sequence
// directly to the banded state (F0; F+k, F-k, Zk, k = 1..n): shift, relax, RF, shift, relax; O(n^2) instead of O(n^3).
// The coefficients and block operators are those of met2_epg.cuh, shared with the parametric fit (met2_param.cu).
#include "met2_host.h"
#include "met2_epg.cuh"

namespace met2 {

__device__ __forceinline__ void epg_decay(double alpha_deg, double T2, double T1, int n, double tau, double scale,
                                          double* out, int out_stride) {
    const EpgCoef<double> c = epg_coef(alpha_deg, T2, T1, tau);
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
