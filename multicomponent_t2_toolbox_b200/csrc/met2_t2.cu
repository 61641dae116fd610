// met2_t2.cu — T2-spectrum estimation and derived maps for a batch of voxels (Steps 3 and 4 of the reference).
//
// Takes over fitting_slice_T2 (motor/motor_recon_met2_real_data.py:113-162) with the solvers it dispatches to —
// nnls (algorithms.py:55), nnls_tik (:262), nnls_x2 (:211-233), nnls_lcurve_wrapper + select_corner (:88-113,150-206),
// BayesReg_nnls (bayesian_interpolation.py:84-126) — the joblib loop around it (motor...:428-441) and the Step-4
// metrics loop (motor...:443-472).
//
// Layout: voxels are counting-sorted by flip-angle index and cut into tiles of <= T2_TILE voxels that share one index.
// A persistent CTA takes a tile, stages that angle's Gram matrix G (n x n) and the band forms of K = L^T L and L in
// shared memory, and its warps pull voxels of the tile one at a time.  One warp owns one voxel from its signal load to
// its outputs: the whole lambda search (Brent / grid) runs in that warp, nothing per-voxel leaves the SM in between.
#include "met2_t2_impl.cuh"

namespace met2 {

// ---------------------------------------------------------------------------------------------- sort by FA index
__global__ void t2_hist_kernel(const int* __restrict__ fa_index, long long V, int nA, int* __restrict__ hist) {
    long long v = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= V) return;
    int f = fa_index[v];
    if (f < 0 || f >= nA) f = 0;   // flagged (and skipped) by the fit kernel
    atomicAdd(&hist[f], 1);
}

// Tiles are handed to the persistent CTAs in list order (atomic counter).  Guided self-scheduling: large tiles first
// (few per-tile barriers and G re-stagings), small tiles for the last `V - switch_off` voxels so that the CTAs run dry
// within a fraction of a large tile's duration of each other.
__global__ void t2_tiles_kernel(const int* __restrict__ hist, int nA, int tile_big, int tile_small, int switch_off,
                                int* __restrict__ bin_start, int* __restrict__ cursor, int* __restrict__ tile_fa,
                                int* __restrict__ tile_start, int* __restrict__ tile_cnt, int* __restrict__ counters) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    int off = 0, nt = 0;
    for (int a = 0; a < nA; ++a) {
        int c = hist[a];
        bin_start[a] = off;
        cursor[a] = 0;
        for (int s = 0; s < c;) {
            const int ts = (off + s < switch_off) ? tile_big : tile_small;
            tile_fa[nt] = a;
            tile_start[nt] = off + s;
            tile_cnt[nt] = (c - s < ts) ? (c - s) : ts;
            s += ts;
            ++nt;
        }
        off += c;
    }
    bin_start[nA] = off;
    counters[0] = nt;
    counters[1] = 0;
}

__global__ void t2_scatter_kernel(const int* __restrict__ fa_index, long long V, int nA,
                                  const int* __restrict__ bin_start, int* __restrict__ cursor, int* __restrict__ perm) {
    long long v = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= V) return;
    int f = fa_index[v];
    if (f < 0 || f >= nA) f = 0;
    int pos = bin_start[f] + atomicAdd(&cursor[f], 1);
    perm[pos] = (int)v;
}

// X2 (nT2 <= 64 columns staged per CTA), T2SPARC, L-curve and BayesReg with MET2_T2_FLAG_ECHO_SPACE run in the reduced
// echo space
bool t2_echo_eligible(const met2_t2_cfg* cfg) {
    if (!(cfg->flags & MET2_T2_FLAG_ECHO_SPACE)) return false;
    if (cfg->method == MET2_REG_X2) return cfg->nT2 <= 64 && !(cfg->flags & MET2_T2_FLAG_COLD_START);
    if (cfg->method == MET2_REG_T2SPARC) return cfg->nT2 <= 128;
    if (cfg->method == MET2_REG_LCURVE || cfg->method == MET2_REG_BAYESREG)
        return cfg->nT2 <= 128 && !(cfg->flags & MET2_T2_FLAG_COLD_START);
    return false;
}

}  // namespace met2

using namespace met2;

static int t2_check_cfg(const met2_t2_cfg* cfg) {
    if (!cfg) return set_error(MET2_ERR_ARG, "met2_t2: cfg is NULL");
    if (cfg->nT2 <= 0 || cfg->nT2 > MET2_MAX_NT2 || cfg->nTE <= 0 || cfg->nTE > MET2_MAX_NTE || cfg->nA <= 0)
        return set_error(MET2_ERR_ARG, "met2_t2: unsupported sizes nT2=%d nTE=%d nA=%d", cfg->nT2, cfg->nTE, cfg->nA);
    if (cfg->method < MET2_REG_NNLS || cfg->method > MET2_REG_BAYESREG)
        return set_error(MET2_ERR_ARG, "met2_t2: unknown method %d", cfg->method);
    if (cfg->method == MET2_REG_LCURVE && (cfg->nLambda < 3 || cfg->nLambda > MET2_MAX_LAMBDAS))
        return set_error(MET2_ERR_ARG, "met2_t2: L-curve needs 3..%d lambdas", MET2_MAX_LAMBDAS);
    // the kernel stages MET2_MAX_LAMBDAS grid values in shared memory and walks gi < nLambda
    if (cfg->method == MET2_REG_GCV && (cfg->flags & MET2_T2_FLAG_GCV_GRID) &&
        (cfg->nLambda < 1 || cfg->nLambda > MET2_MAX_LAMBDAS))
        return set_error(MET2_ERR_ARG, "met2_t2: GCV grid needs 1..%d lambdas, got %d", MET2_MAX_LAMBDAS, cfg->nLambda);
    if ((cfg->flags & MET2_T2_FLAG_ECHO_SPACE) && cfg->echo_rank != 0 && cfg->echo_rank != MET2_ECHO_RANK &&
        cfg->echo_rank != MET2_ECHO_RANK_SMALL)
        return set_error(MET2_ERR_ARG, "met2_t2: echo_rank must be 0, %d or %d, got %d", MET2_ECHO_RANK_SMALL, MET2_ECHO_RANK,
                         cfg->echo_rank);
    return MET2_OK;
}

// number of shared full-set factor tables this configuration builds (0: none)
static int t2_full_tables(const met2_t2_cfg* cfg) {
    if (cfg->flags & MET2_T2_FLAG_COLD_START) return 0;
    if (t2_echo_eligible(cfg)) return 0;
    if (cfg->method == MET2_REG_X2 && (cfg->flags & MET2_T2_FLAG_FULL_START)) return T2_NTAB_X2;
    if (cfg->method == MET2_REG_BAYESREG) return T2_NTAB_BAYES;
    return 0;
}

template <int NS>
static int t2_launch_full_factors(const T2Args& A, int ntab, const double* G, const double* kband, double* tfull,
                                  double* lam_tab, cudaStream_t st) {
    const int n = A.cfg.nT2;
    const size_t smem = sizeof(double) * (size_t)Slots<NS>::doubles(n);
    cudaError_t e = cudaFuncSetAttribute(t2_full_factors_kernel<NS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return set_error(MET2_ERR_CUDA, "t2_full_factors attr: %s", cudaGetErrorString(e));
    MET2_LAUNCH(ntab * A.cfg.nA, 32, smem, st, t2_full_factors_kernel<NS>)(G, kband, n, A.cfg.nA, A.cfg.brent_lo, A.cfg.brent_hi,
                                                                     A.cfg.brent_xatol, A.cfg.maxfun,
                                                                     A.cfg.method == MET2_REG_BAYESREG ? 1 : 0, tfull, lam_tab);
    count_launch();
    return check_launch("t2_full_factors_kernel");
}

extern "C" int64_t met2_t2_workspace_bytes(int64_t V, const met2_t2_cfg* cfg) {
    if (t2_check_cfg(cfg) || V < 0) return -1;
    T2Geom g = t2_geometry_any(V, cfg, read_overrides());
    size_t b = 0;
    b += align256(sizeof(int) * (size_t)cfg->nA) * 2;
    b += align256(sizeof(int) * (size_t)(cfg->nA + 1));
    b += align256(sizeof(int) * (size_t)V);
    b += align256(sizeof(int) * (size_t)g.max_tiles) * 3;
    b += align256(sizeof(int) * 4);
    if (t2_full_tables(cfg))
        b += align256(sizeof(double) * T2_NTAB_MAX) +
             align256(sizeof(double) * (size_t)t2_full_tables(cfg) * cfg->nA * tri(cfg->nT2));
    return (int64_t)b + 256;
}

static int t2_fit_impl(const double* sig, const int32_t* fa_index, int64_t V, const met2_t2_cfg* cfg,
                       const double* dic, const double* dicT, const double* G, const double* kband,
                       const double* lambdas, const double* logT2, const uint8_t* comp, const double* red_basis,
                       const double* red_coef, double* fsol, double* est_signal, double* reg, double* maps,
                       uint32_t* status, void* workspace, void* stream) {
    int rc = t2_check_cfg(cfg);
    if (rc) return rc;
    if (V < 0 || !sig || !fa_index || !dic || !dicT || !G || !logT2 || !comp || !fsol || !est_signal || !reg || !maps ||
        !status || !workspace)
        return set_error(MET2_ERR_ARG, "met2_t2_fit: NULL argument");
    if (cfg->method != MET2_REG_NNLS && !kband)
        return set_error(MET2_ERR_ARG, "met2_t2_fit: regularised methods need kband (met2_gram_tables)");
    if (cfg->method == MET2_REG_LCURVE && !lambdas) return set_error(MET2_ERR_ARG, "met2_t2_fit: L-curve needs lambdas");
    if (cfg->method == MET2_REG_GCV && (cfg->flags & MET2_T2_FLAG_GCV_GRID) && !lambdas)
        return set_error(MET2_ERR_ARG, "met2_t2_fit: the GCV grid mode needs lambdas");
    if (t2_echo_eligible(cfg) && (!red_basis || !red_coef))
        return set_error(MET2_ERR_ARG, "met2_t2_fit: MET2_T2_FLAG_ECHO_SPACE needs the reduced echo basis (met2_echo_basis)");
    if (V == 0) return MET2_OK;
    if (V > 0x7fffffffLL) return set_error(MET2_ERR_ARG, "met2_t2_fit: V too large for one call");
    cudaStream_t st = (cudaStream_t)stream;
    const Overrides ov = read_overrides();
    T2Geom g = t2_geometry_any(V, cfg, ov);
    T2Args A;
    A.sig = sig; A.fa_index = fa_index; A.V = V; A.cfg = *cfg;
    A.dic = dic; A.dicT = dicT; A.G = G; A.kband = kband; A.lambdas = lambdas; A.logT2 = logT2; A.comp = comp;
    A.fsol = fsol; A.est = est_signal; A.reg = reg; A.maps = maps; A.status = status;
    A.red_basis = red_basis; A.red_coef = red_coef;
    unsigned char* w = reinterpret_cast<unsigned char*>(((uintptr_t)workspace + 255) & ~(uintptr_t)255);
    A.hist = reinterpret_cast<int*>(w);        w += align256(sizeof(int) * (size_t)cfg->nA);
    A.cursor = reinterpret_cast<int*>(w);      w += align256(sizeof(int) * (size_t)cfg->nA);
    A.bin_start = reinterpret_cast<int*>(w);   w += align256(sizeof(int) * (size_t)(cfg->nA + 1));
    A.perm = reinterpret_cast<int*>(w);        w += align256(sizeof(int) * (size_t)V);
    A.tile_fa = reinterpret_cast<int*>(w);     w += align256(sizeof(int) * (size_t)g.max_tiles);
    A.tile_start = reinterpret_cast<int*>(w);  w += align256(sizeof(int) * (size_t)g.max_tiles);
    A.tile_cnt = reinterpret_cast<int*>(w);    w += align256(sizeof(int) * (size_t)g.max_tiles);
    A.counters = reinterpret_cast<int*>(w);  w += align256(sizeof(int) * 4);
    A.pmax = g.pmax;
    A.warps = g.warps;
    A.tfull = nullptr;
    A.lam_tab = nullptr;
    A.ntab = 0;
    A.ntab_use = 0;
    A.lcurve_switch = ov.lcurve_switch_set ? ov.lcurve_switch : T2_LCURVE_SWITCH;
    if (const int ntab = t2_full_tables(cfg)) {
        double* lam_tab = reinterpret_cast<double*>(w);  w += align256(sizeof(double) * T2_NTAB_MAX);
        double* tfull = reinterpret_cast<double*>(w);
        const int ns = (cfg->nT2 + 31) / 32;
        if (ns <= 2) rc = t2_launch_full_factors<2>(A, ntab, G, kband, tfull, lam_tab, st);
        else if (ns == 3) rc = t2_launch_full_factors<3>(A, ntab, G, kband, tfull, lam_tab, st);
        else rc = t2_launch_full_factors<4>(A, ntab, G, kband, tfull, lam_tab, st);
        if (rc) return rc;
        A.ntab = ntab;
        // full-set starts of the NNLS solves: X2 only (measured; for BayesReg the tables serve the evidence)
        A.ntab_use = (cfg->method == MET2_REG_X2) ? ntab : 0;
        A.tfull = tfull;
        A.lam_tab = lam_tab;
    }
    cudaError_t e = cudaMemsetAsync(A.hist, 0, sizeof(int) * (size_t)cfg->nA, st);
    if (e != cudaSuccess) return set_error(MET2_ERR_CUDA, "memset hist: %s", cudaGetErrorString(e));
    const int tb = 256;
    const unsigned nb = (unsigned)((V + tb - 1) / tb);
    MET2_LAUNCH(nb, tb, 0, st, t2_hist_kernel)(fa_index, V, cfg->nA, A.hist);
    count_launch();
    if ((rc = check_launch("t2_hist_kernel"))) return rc;
    MET2_LAUNCH(1, 32, 0, st, t2_tiles_kernel)(A.hist, cfg->nA, g.tile_big, g.tile_small, g.switch_off, A.bin_start, A.cursor,
                                      A.tile_fa, A.tile_start, A.tile_cnt, A.counters);
    count_launch();
    if ((rc = check_launch("t2_tiles_kernel"))) return rc;
    MET2_LAUNCH(nb, tb, 0, st, t2_scatter_kernel)(fa_index, V, cfg->nA, A.bin_start, A.cursor, A.perm);
    count_launch();
    if ((rc = check_launch("t2_scatter_kernel"))) return rc;
    if (t2_echo_eligible(cfg)) {
        const bool small = (cfg->echo_rank == MET2_ECHO_RANK_SMALL);
        if (cfg->method == MET2_REG_LCURVE || cfg->method == MET2_REG_BAYESREG)
            return small ? t2_launch_echo_reg_r16(A, ov, st) : t2_launch_echo_reg_r24(A, ov, st);
        return small ? t2_launch_echo_r16(A, ov, st) : t2_launch_echo_r24(A, ov, st);
    }
    switch (cfg->method) {
        case MET2_REG_NNLS: return t2_launch_nnls(A, g, st);
        case MET2_REG_T2SPARC: return t2_launch_t2sparc(A, g, st);
        case MET2_REG_X2: return t2_launch_x2(A, g, st);
        case MET2_REG_LCURVE: return t2_launch_lcurve(A, g, st);
        case MET2_REG_BAYESREG: return t2_launch_bayesreg(A, g, st);
        case MET2_REG_GCV: return t2_launch_gcv(A, g, st);
        default: return set_error(MET2_ERR_UNSUPPORTED, "met2_t2_fit: method %d not implemented", cfg->method);
    }
}

extern "C" int met2_t2_fit(const double* sig, const int32_t* fa_index, int64_t V, const met2_t2_cfg* cfg,
                           const double* dic, const double* dicT, const double* G, const double* kband,
                           const double* lambdas, const double* logT2, const uint8_t* comp, double* fsol,
                           double* est_signal, double* reg, double* maps, uint32_t* status, void* workspace,
                           void* stream) {
    return t2_fit_impl(sig, fa_index, V, cfg, dic, dicT, G, kband, lambdas, logT2, comp, nullptr, nullptr, fsol,
                       est_signal, reg, maps, status, workspace, stream);
}

extern "C" int met2_t2_fit_echo(const double* sig, const int32_t* fa_index, int64_t V, const met2_t2_cfg* cfg,
                                const double* dic, const double* dicT, const double* G, const double* kband,
                                const double* lambdas, const double* logT2, const uint8_t* comp,
                                const double* red_basis, const double* red_coef, double* fsol, double* est_signal,
                                double* reg, double* maps, uint32_t* status, void* workspace, void* stream) {
    return t2_fit_impl(sig, fa_index, V, cfg, dic, dicT, G, kband, lambdas, logT2, comp, red_basis, red_coef, fsol,
                       est_signal, reg, maps, status, workspace, stream);
}
