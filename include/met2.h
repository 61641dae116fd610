/* met2.h — C ABI of libmet2.so: the B200 (sm_100a) implementation of the per-voxel MET2 inverse-problem path.
 *
 * The reference (ejcanalesr/multicomponent-T2-toolbox) is pure Python and has no FFI; the boundary this library
 * replaces is the set of Python call signatures listed in SURVEY.md §8(b).  Each entry point below names the
 * reference interface (file:line under the reference tree) whose work it takes over.
 *
 * Conventions
 *   - every array argument is a DEVICE pointer to a contiguous C-order array (float64 unless said otherwise) that the
 *     caller owns; the library never allocates or frees caller buffers.  Scratch space is passed in as `workspace`
 *     (size from the matching *_workspace_bytes call; 256-byte aligned device memory).
 *   - all work is enqueued on `stream` (a cudaStream_t passed as void*; NULL = default stream) and is asynchronous;
 *     the caller synchronises.  One call at a time per stream.
 *   - return value 0 = success, negative = error (message from met2_last_error(), thread-local).  No exception and
 *     no abort crosses the ABI.  Per-voxel conditions never fail the batch: they are reported as bit flags in
 *     `status[v]` (MET2_ST_*), and a skipped voxel gets all-zero outputs exactly like the reference's zero-initialised
 *     arrays (motor/motor_recon_met2_real_data.py:115-117,191-202).
 *   - there is no CPU fallback: without a CUDA device every compute entry point returns MET2_ERR_CUDA.
 */
#ifndef MET2_H_
#define MET2_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MET2_VERSION 120 /* 0.1.2: met2_t2_cfg.echo_rank, met2_echo_rank; L-curve / BayesReg in the reduced echo space */

/* error codes */
#define MET2_OK 0
#define MET2_ERR_ARG (-1)   /* invalid argument (sizes out of the supported range, NULL pointer, bad enum) */
#define MET2_ERR_CUDA (-2)  /* CUDA runtime error (message holds cudaGetErrorString) */
#define MET2_ERR_UNSUPPORTED (-3)

/* supported sizes */
#define MET2_MAX_NT2 128 /* T2 bins (reference: 60, or 96 for T2SPARC; config 4 uses 100) */
#define MET2_MAX_NTE 64  /* echoes (reference data: 32; config 4 uses 48) */
#define MET2_MAX_KNOTS 32
#define MET2_MAX_LAMBDAS 64
#define MET2_ECHO_RANK 24       /* rows of the reduced echo space (met2_echo_basis, met2_t2_fit_echo): exact to the rounding
                                   of the dictionary's own entries for every protocol met so far */
#define MET2_ECHO_RANK_SMALL 16 /* the smaller rank the echo-space kernels are also built for: valid when the residual of
                                   the rank-16 reduction (`tail` of met2_echo_basis) is below 4e-12, as for the
                                   reference's 32-echo protocol (1.6e-12); 19 % faster (met2_t2_cfg.echo_rank) */

/* per-voxel status bits */
#define MET2_ST_SKIPPED 1u      /* sum(M) <= 0 or M[0] <= 0: voxel not fitted (fa_estimation.py:100, motor...:124,131) */
#define MET2_ST_NONFINITE 2u    /* NaN/Inf in the signal (the reference raises ValueError, algorithms.py:56) */
#define MET2_ST_ITMAX 4u        /* a Lawson-Hanson solve hit itmax = 3n (ignored by the reference, algorithms.py:79-81) */
#define MET2_ST_SSE_ZERO 8u     /* X2: plain-NNLS residual is exactly 0 -> NaN objective (algorithms.py:231) */
#define MET2_ST_ECHO_BAD_L 32u  /* MET2_T2_FLAG_ECHO_SPACE given with a non-diagonal L: voxel skipped */
#define MET2_ST_NOT_PD 16u      /* BayesReg: beta*B + beta*x*K not positive definite (reference: LinAlgError) */
#define MET2_ST_AT_BOUND 64u    /* met2_param_fit: a fitted T2 or the flip angle ends on its box (informational) */
#define MET2_ST_MM_CAP 128u     /* met2_rician_fit: the MM iteration ran max_iter solves without meeting tol */
#define MET2_ST_BAD_SIGMA 256u  /* met2_rician_fit: the noise sigma is NaN, +-Inf or negative (voxel skipped) */

/* flip-angle search methods: run_real_data_script.py --FA_method */
#define MET2_FA_BRUTE_FORCE 0
#define MET2_FA_SPLINE 1

/* regularisation methods: run_real_data_script.py --reg_method */
#define MET2_REG_NNLS 0
#define MET2_REG_T2SPARC 1
#define MET2_REG_X2 2
#define MET2_REG_LCURVE 3
#define MET2_REG_GCV 4
#define MET2_REG_BAYESREG 5

typedef struct met2_fa_cfg {
    int32_t method;       /* MET2_FA_* */
    int32_t nTE, nT2;     /* echoes, T2 bins */
    int32_t nA;           /* flip angles of the fine grid (91 brute-force / 273 spline; motor...:231-245) */
    int32_t nKnots;       /* spline only: angles of the coarse dictionary (15) */
    int32_t final_solve;  /* 1: also solve NNLS at the chosen angle -> km, fsol_sum (fa_estimation.py:61-65,84-86) */
    double brent_lo, brent_hi, brent_xatol; /* spline: minimize_scalar(method='Bounded') bounds=(90,180), 1e-5 */
    int32_t brent_maxfun;                   /* 500 */
    int32_t reserved;
} met2_fa_cfg;

/* met2_t2_cfg.flags */
#define MET2_T2_FLAG_REG_IS_LAMBDA 1 /* reg[v] = the selected lambda for every method (default: what the orchestrator
                                        stores, motor...:134-155: 0 | 1.8 | k_est for X2 | lambda) */
#define MET2_T2_FLAG_NO_NORMALISE 2  /* fit M as given instead of M / M[0] (per-voxel API of algorithms.py) */
#define MET2_T2_FLAG_GCV_EVAL 8      /* GCV only: no search; solve at lambda_fixed and return the GCV objective
                                        (algorithms.py:285-296) in reg[v] — for objective-level parity tests; bits
                                        16-23 of status[v] then hold the rank the truncated pseudo-inverse kept
                                        (the `rank` of the reference's np.linalg.lstsq) */
#define MET2_T2_FLAG_GCV_GRID 32     /* GCV only (extension, BASELINE.json configs[2]): instead of Brent, evaluate the
                                        objective of algorithms.py:285-296 on `lambdas[0..nLambda)` and take the arg-min */
#define MET2_T2_FLAG_FULL_START 16    /* X2: start the solves at Brent's first (voxel-independent) abscissae from the full
                                        column set, with inverse-Cholesky factors shared per flip angle
                                        (worth it when L = I; same minimiser) */
#define MET2_T2_FLAG_ECHO_SPACE 64    /* X2 (nT2 <= 64), T2SPARC, L-curve and BayesReg (nT2 <= 128) with a DIAGONAL L (I,
                                        InvT2; asserted by the caller): Tikhonov solves in the reduced echo space (16 x 16
                                        or 24 x 24 factor per voxel, csrc/met2_t2_echo_impl.cuh, met2_t2_echo_reg_impl.cuh)
                                        instead of the Gram domain (nT2 x nT2).  Needs the tables of met2_echo_basis ->
                                        call met2_t2_fit_echo with cfg.echo_rank = their R.  A non-diagonal L skips every
                                        voxel with MET2_ST_ECHO_BAD_L; every other method ignores the flag.  Same
                                        minimiser as the Gram-domain path; measured 1.4-3.6x faster (profiles/r02_ab_*),
                                        which is why batched.Met2Plan sets it by default for these methods */
#define MET2_T2_FLAG_COLD_START 4    /* start every NNLS of a lambda search from the empty set like the reference,
                                        instead of warm-starting from the previous solution (same minimiser) */

typedef struct met2_t2_cfg {
    int32_t method;   /* MET2_REG_* */
    int32_t nTE, nT2, nA;
    int32_t nLambda;  /* L-curve grid size (50) */
    int32_t maxfun;   /* Brent evaluation cap: X2/GCV 300, BayesReg 200 */
    double factor;    /* X2 chi-square factor 1.02 (motor...:141) */
    double lambda_fixed; /* T2SPARC 1.8 (motor...:138) */
    double brent_lo, brent_hi, brent_xatol; /* X2 [0,10]; GCV [1e-8,10]; BayesReg [1e-8,2]; xtol 1e-5 */
    double log_det_L;    /* BayesReg: log(det(L)) (bayesian_interpolation.py:100,123); -inf for L2 */
    int32_t flags;       /* MET2_T2_FLAG_* */
    int32_t echo_rank;   /* MET2_T2_FLAG_ECHO_SPACE: the R the tables of met2_echo_basis were built with — MET2_ECHO_RANK
                            (also 0) or MET2_ECHO_RANK_SMALL; ignored otherwise */
} met2_t2_cfg;

/* Replaces epg/epg.py:155 create_Dic_3D (-> :47 create_met2_design_matrix_epg -> :64 epg_signal).
 * dic  [nA][nTE][nT2]  (the reference's Dic_3D[:, :, a] slices made contiguous) and
 * dicT [nA][nT2][nTE]  (same numbers transposed, for coalesced residual evaluation).  Either may be NULL. */
int met2_epg_dictionary(const double* alphas_deg, int nA, const double* T2s, const double* T1s, int nT2, int nTE,
                        double tau_ms, double TR_ms, double* dic, double* dicT, void* stream);

/* EPG decay curves for arbitrary (alpha, T2, T1) triples: sig[N][nTE] without the (1-exp(-TR/T1)) factor.
 * Same kernel as the dictionary; used by the synthetic phantom generator (epg/epg.py:64 epg_signal). */
int met2_epg_signals(const double* alphas_deg, const double* T2s, const double* T1s, int64_t N, int nTE, double tau_ms,
                     double* sig, void* stream);

/* Gram tables of the dictionary, G[a] = D_a^T D_a  ([nA][nT2][nT2]), and the 5-band form of K = L^T L
 * (kband[10][nT2]: rows 0..4 kband[d][c] = K[c+d-2][c], rows 5..9 the row-band form of L itself, kband[5+d][r] = L[r][r+d-2]) for the Tikhonov term of algorithms.py:262-269 (A = [D; sqrt(lambda) L]).
 * L is the dense [nT2][nT2] matrix of motor...:86-111,254-273; *band_err (device int, may be NULL) is set to 1 if
 * L^T L has an entry outside the five central diagonals (not the case for I, L1, L2, InvT2).  L/kband may be NULL. */
int met2_gram_tables(const double* dic, int nA, int nTE, int nT2, const double* L, double* G, double* kband,
                     int32_t* band_err, void* stream);

/* Replaces the Step-2 joblib loop (motor...:349-373) over fitting_slice_FA_brute_force (fa_estimation.py:92) /
 * fitting_slice_FA_spline_method (:35) and their per-voxel body compute_optimal_FA (:74).
 * sig [V][nTE] raw signals of the voxels to fit (mask already applied by the caller).
 * Search dictionary = (dic_s, dicT_s, G_s) with cfg->nKnots angles for the spline method, or the fine dictionary
 * itself for brute force (pass the same pointers).  alphas [nA] fine grid (deg), knots [nKnots].
 * Outputs: fa_index [V] int32, fa_deg [V], km [V] (sum of the NNLS spectrum at the chosen angle),
 * fsol_sum [nT2] (sum over voxels of those spectra; feeds mean_T2_dist, motor...:362,370), status [V] uint32. */
int64_t met2_fa_workspace_bytes(int64_t V, const met2_fa_cfg* cfg);
int met2_fa_fit(const double* sig, int64_t V, const met2_fa_cfg* cfg, const double* dic, const double* dicT,
                const double* G, const double* alphas, const double* dic_s, const double* dicT_s, const double* G_s,
                const double* knots, int32_t* fa_index, double* fa_deg, double* km, double* fsol_sum, uint32_t* status,
                void* workspace, void* stream);

/* Replaces the Step-3 joblib loop (motor...:428-441) over fitting_slice_T2 (motor...:113-162) with its solvers
 * nnls / nnls_tik / nnls_x2 / nnls_lcurve_wrapper / nnls_gcv (intravoxel_algorithms/algorithms.py:55-296) and
 * BayesReg_nnls (intravoxel_algorithms/bayesian_interpolation.py:84-126), and the Step-4 metrics loop (motor...:443-472).
 * sig [V][nTE] raw signals; fa_index [V]; kband from met2_gram_tables; lambdas [nLambda] (L-curve grid);
 * logT2 [nT2]; comp [nT2] uint8 bit mask per T2 bin: 1 = myelin (ind_m), 2 = intra/extra (ind_t), 4 = free water (ind_csf).
 * Outputs: fsol [V][nT2], est_signal [V][nTE], reg [V] (motor...:153: 0 | 1.8 | k_est | lambda),
 * maps [V][6] = MWF, IEWF, FWF, T2_M, T2_IE, TWC, status [V]. */
int64_t met2_t2_workspace_bytes(int64_t V, const met2_t2_cfg* cfg);
int met2_t2_fit(const double* sig, const int32_t* fa_index, int64_t V, const met2_t2_cfg* cfg, const double* dic,
                const double* dicT, const double* G, const double* kband, const double* lambdas, const double* logT2,
                const uint8_t* comp, double* fsol, double* est_signal, double* reg, double* maps, uint32_t* status,
                void* workspace, void* stream);

/* Reduced echo basis of the dictionary (once per reconstruction).  The EPG decay curves of one flip angle are
 * numerically of rank ~20 whatever nTE is: D_a = U_a C_a to the rounding of D_a's own entries, with U_a [nTE][R]
 * orthonormal and C_a = U_a^T D_a (column-pivoted Gram-Schmidt, csrc/met2_basis.cu).
 * basis [nA][nTE][R], coef [nA][nT2][R] (C_a[e][j] stored at [j][e]), tail [nA] = max_j |d_j - U C_j| / max_j |d_j|
 * per angle (may be NULL): the measured residual of the reduction, which the caller checks against its tolerance
 * (batched.ECHO_TAIL_MAX: 1e-15 at rank 24, 4e-12 at rank 16) before using the echo-space kernels.  For met2_t2_fit_echo R
 * must be MET2_ECHO_RANK or MET2_ECHO_RANK_SMALL (met2_echo_rank) and be passed in cfg.echo_rank. */
int met2_echo_basis(const double* dic, int nA, int nTE, int nT2, int R, double* basis, double* coef, double* tail,
                    void* stream);

/* met2_t2_fit with the tables of met2_echo_basis: required when cfg->flags has MET2_T2_FLAG_ECHO_SPACE (the X2 / T2SPARC /
 * L-curve / BayesReg Tikhonov solves then run in the reduced echo space); otherwise identical to met2_t2_fit. */
int met2_t2_fit_echo(const double* sig, const int32_t* fa_index, int64_t V, const met2_t2_cfg* cfg, const double* dic,
                     const double* dicT, const double* G, const double* kband, const double* lambdas,
                     const double* logT2, const uint8_t* comp, const double* red_basis, const double* red_coef,
                     double* fsol, double* est_signal, double* reg, double* maps, uint32_t* status, void* workspace,
                     void* stream);

/* FA-stage preprocessing: replaces `filt.gaussian_filter(data[:, :, :, c], 2.0, 0)` per echo (motor...:336-346;
 * scipy.ndimage semantics: mode 'reflect', symmetric kernel `weights[2*radius+1]`, radius = int(4 sigma + 0.5)).
 * vol/out/tmp are [nx][ny][nz][nt] C-order device arrays; out and tmp must not alias vol. */
int met2_gaussian_smooth(const double* vol, int nx, int ny, int nz, int nt, const double* weights, int radius,
                         double* out, double* tmp, void* stream);

/* Per-segment mean signal and mean kernel: the inputs of the reference's mean-spectrum diagnostics
 * (motor/motor_recon_met2_real_data.py:377-403, one segment: mask == 1) and of its ROI-based estimator
 * (motor/motor_recon_met2_real_data_ROI.py:405-445, one segment per ROI label), which both walk the whole volume in a
 * Python triple loop:  total_signal = mean of data[v, :],  total_Kernel = mean of Dic_3D[:, :, FA_index[v]]  over the
 * voxels of the segment.  label [V] int32 segment id in [0, nSeg) (anything else: voxel in no segment).
 * Outputs: mean_signal [nSeg][nTE], mean_kernel [nSeg][nTE][nT2] (the layout of `dic`, usable as an nSeg-"angle"
 * dictionary for met2_t2_fit), counts [nSeg] int32.  An empty segment gives NaN (the reference divides by nv = 0). */
int64_t met2_segment_workspace_bytes(int nSeg, int nA);
int met2_segment_means(const double* sig, const int32_t* fa_index, const int32_t* label, int64_t V, int nTE, int nT2,
                       int nA, int nSeg, const double* dic, double* mean_signal, double* mean_kernel, int32_t* counts,
                       void* workspace, void* stream);

/* Optional Step-1 preprocessing: replaces the NESMA loop of motor/motor_recon_met2_real_data.py:305-333.  For every
 * voxel with mask == 1: RE_p = 100 * sum_t |s_p(t) - s(t)| / sum_t s(t) over the window [c - hw, c + hw) per axis
 * (clipped to the volume; hw = path_size = 6), out = mean of the s_p with RE_p < threshold_percent (2.5).  Voxels with
 * mask != 1 get zeros.  vol/out [nx][ny][nz][nt] C-order, mask [nx][ny][nz] int32, tmp: nx*ny*nz*nt doubles of
 * scratch (echo-major copy of vol); out and tmp must not alias vol. */
int met2_nesma_filter(const double* vol, const int32_t* mask, int nx, int ny, int nz, int nt, int half_window,
                      double threshold_percent, double* out, double* tmp, void* stream);

/* Optional Step-1 preprocessing, --denoise TV (motor/motor_recon_met2_real_data.py:293-303): per echo volume
 * vol[..., t] with its axes of size 1 dropped (np.squeeze), scikit-image's noise estimate and Chambolle TV filter.
 * vol/out [nx][ny][nz][nt] C-order; out must not alias vol.  At least one spatial axis must be longer than 1.
 *
 * met2_noise_sigma: sigma[t] = median(|c| over the nonzero c) / norm.ppf(0.75), c = the single-level db2 detail band
 * (PyWavelets 'symmetric' mode, the high-pass along every remaining axis); NaN if a coefficient is NaN or none is
 * nonzero (skimage.restoration.estimate_sigma(vol, channel_axis=None)).  sigma [nt], device.
 *
 * met2_tv_chambolle: skimage.restoration.denoise_tv_chambolle(vol, weight[t], eps, max_iter) per echo (the nd-Chambolle
 * iteration with tau = 1 / (2 ndim), stopping when |E_prev - E| < eps * E_init).  weight [nt] is a device array, so that
 * 2 * sigma can be passed without a round trip; iterations [nt] int32 receives the number of iterations run per echo.
 * Both are bitwise equal to the NumPy restatement in tests/tv_oracle.py (energy sums in NumPy's pairwise order). */
int64_t met2_noise_sigma_workspace_bytes(int nx, int ny, int nz, int nt);
int met2_noise_sigma(const double* vol, int nx, int ny, int nz, int nt, double* sigma, void* workspace, void* stream);
int64_t met2_tv_workspace_bytes(int nx, int ny, int nz, int nt);
int met2_tv_chambolle(const double* vol, int nx, int ny, int nz, int nt, const double* weight, double eps, int max_iter,
                      double* out, int32_t* iterations, void* workspace, void* stream);

/* Optional Step-1 preprocessing (no counterpart in the reference): Marchenko-Pastur PCA denoising (Veraart et al. 2016,
 * MRtrix3's dwidenoise) with a per-voxel noise map.  Definition in csrc/met2_mppca.cu; bitwise equal to the NumPy
 * restatement in tests/mppca_oracle.py.  For every voxel with mask == 1: PCA of the (2r + 1)^3 window (shifted, not
 * shrunk, at the volume's edges), Marchenko-Pastur split of the eigenvalues into noise and signal, and the centre voxel
 * rebuilt from the signal components.  vol/out [nx][ny][nz][nt] C-order (out must not alias vol), mask [nx][ny][nz]
 * int32; outputs out, sigma [nx][ny][nz] (the noise standard deviation) and n_signal [nx][ny][nz] int32.  Voxels with
 * mask != 1 get zeros; a window holding a non-finite sample gives out = the input, sigma = NaN, n_signal = -1.
 * nt <= MET2_MAX_NTE, r >= 1 and at least 2 samples per window, else MET2_ERR_ARG before anything is enqueued; a mask
 * with no voxel set is not an error (all outputs zero). */
int64_t met2_mppca_workspace_bytes(int nx, int ny, int nz, int nt, int r);
int met2_mppca(const double* vol, const int32_t* mask, int nx, int ny, int nz, int nt, int r, double* out, double* sigma,
               int32_t* n_signal, void* workspace, void* stream);

/* Optional preprocessing after Step 1 (no counterpart in the reference): Gibbs-ringing removal by local subvoxel shifts
 * (Kellner et al. 2016, MRtrix3's mrdegibbs, basic 2-D mode; partial-Fourier data are out of scope) on every in-plane
 * slice vol[:, :, z, t].  Definition in csrc/met2_degibbs.cu; bitwise equal to the NumPy restatement in
 * tests/degibbs_oracle.py.  vol/out [nx][ny][nz][nt] C-order float64 (out must not alias vol).  nsh shifts per half
 * pixel (MRtrix: 20), TV window minW..maxW (MRtrix: 1..3).  1 <= nx, ny <= 256, nsh >= 1, 0 <= minW <= maxW,
 * 2 maxW < nx and ny, and (2 nsh + 33) * 8 * max(nx, ny) bytes <= 227 KB (nsh <= 40 at 256), else MET2_ERR_ARG before
 * anything is enqueued.
 * met2_degibbs_tables writes the n * (2 nsh + 4) doubles of the tables of in-plane size n (cos[n], sin[n],
 * 1 + cos(2 pi fftfreq)[n], the interpolation kernels h[2 nsh + 1][n]) to host_out unless it is NULL, and returns that
 * count (MET2_ERR_ARG for n outside 1..256 or nsh outside 1..1024).  The kernels build the same bits on the device. */
int64_t met2_degibbs_tables(int n, int nsh, double* host_out);
int64_t met2_degibbs_workspace_bytes(int nx, int ny, int nz, int nt, int nsh, int minW, int maxW);
int met2_degibbs(const double* vol, int nx, int ny, int nz, int nt, int nsh, int minW, int maxW, double* out,
                 void* workspace, void* stream);

/* Per-voxel bootstrap uncertainty of the six maps (no counterpart in the reference).  Definition in
 * csrc/met2_boot.cu; both calls are bitwise equal to the NumPy restatement in tests/boot_oracle.py.
 *
 * met2_boot_resample: wild-bootstrap replicates with Rademacher signs, rows r = v*B + b of rep_sig [V*B][nTE]:
 * s*_e = est_e +/- (sig_e - est_e), the sign from bit e of splitmix64(seed, (voxel_offset + v)*B + b), so that a voxel's
 * replicates depend only on its position in the whole voxel list.  sig [V][nTE] is the signal the point fit used,
 * est_signal [V][nTE] its fitted signal, fa_index [V] its flip-angle index; rep_fa_index [V*B] repeats it (the FA is
 * held at the point estimate).  1 <= B <= 1024, 1 <= nTE <= MET2_MAX_NTE.
 *
 * met2_boot_summary: over the replicates b of voxel v whose rep_status lacks MET2_ST_SKIPPED (n_valid [V] of them), per
 * map (columns of rep_maps [V*B][6], the `maps` of met2_t2_fit): stats [V][6][4] = mean, sd (ddof 1), 2.5th and 97.5th
 * percentile (numpy's 'linear' method).  n_valid = 0: zeros; a NaN among a map's values: that map's four numbers NaN.
 *
 * Both: V = 0 is a no-op; bad arguments return MET2_ERR_ARG before anything is enqueued. */
int met2_boot_resample(const double* sig, const double* est_signal, const int32_t* fa_index, int64_t V, int nTE,
                       int B, uint64_t seed, int64_t voxel_offset, double* rep_sig, int32_t* rep_fa_index,
                       void* stream);
int met2_boot_summary(const double* rep_maps, const uint32_t* rep_status, int64_t V, int B, double* stats,
                      int32_t* n_valid, void* stream);

/* Spatially regularised spectrum fitting (no counterpart in the reference; the reference's unused prior-spectrum
 * argument points the same way).  Definition in csrc/met2_spatial.cu; the NumPy restatement is tests/spatial_oracle.py.
 * Normalised units: x [V][nT2] holds fsol / sig[0] of the point fit (met2_t2_fit) and is updated in place.
 *
 * met2_spatial_sweep: one half-sweep of red-black block updates, for the voxels vox [Vc] (positions in 0..V-1, all of
 * one colour): x_v <- argmin_{x >= 0} ||D_a x - y_v||^2 + lam_v ||L x||^2 + mu n_v ||x - p_v||^2, with y_v = sig_v /
 * sig_v[0], a = fa_index[v], p_v the mean of the rows x_q of its n_v neighbours q = nbr[v][0..6) (int32, -1 = none).
 * lam [V] is the point fit's lambda (reg under MET2_T2_FLAG_REG_IS_LAMBDA); G, dicT, kband as for met2_t2_fit.
 * status [V]: voxels with MET2_ST_SKIPPED are left alone; a solve that hits itmax ORs MET2_ST_ITMAX.
 *
 * met2_spatial_finish: fsol = x sig[0], est_signal = D_a x sig[0] and maps [V][6] as met2_t2_fit computes them; voxels
 * with MET2_ST_SKIPPED in status get met2_t2_fit's outputs for a skipped voxel.
 *
 * Both: gram-domain sizes of met2_t2_fit (nT2 <= 128, nTE <= 64), V < 2^31; mu must be finite and >= 0; V (or Vc) = 0
 * is a no-op; bad arguments return MET2_ERR_ARG before anything is enqueued. */
int met2_spatial_sweep(const double* sig, const int32_t* fa_index, const double* lam, const int32_t* nbr,
                       const int32_t* vox, int64_t Vc, int64_t V, int nTE, int nT2, int nA, const double* G,
                       const double* dicT, const double* kband, double mu, double* x, uint32_t* status, void* stream);
int met2_spatial_finish(const double* sig, const int32_t* fa_index, const uint32_t* status, const double* x,
                        int64_t V, int nTE, int nT2, int nA, const double* dicT, const double* logT2,
                        const uint8_t* comp, double* fsol, double* est_signal, double* maps, void* stream);

/* Three-pool parametric T2 fit (no counterpart in the reference): bounded Levenberg-Marquardt over the amplitudes and
 * continuous T2s of a myelin, an intra/extra-cellular and a free-water pool, each an EPG decay curve of the dictionary's
 * recurrence, sharing one continuous refocusing angle.  Definition and defaults in csrc/met2_param.cu; the NumPy
 * restatement is tests/param_oracle.py.
 * Inputs are the point fit's: sig [V][nTE] raw signals, fa_deg [V] (met2_fa_fit), fsol [V][nT2] and status [V]
 * (met2_t2_fit); logT2 [nT2] and comp [nT2] as for met2_t2_fit.  Voxels with MET2_ST_SKIPPED or MET2_ST_NONFINITE get
 * all-zero outputs.  Outputs: params [V][7] = the three amplitudes (raw units), the three T2s (ms) and the flip angle
 * (deg); maps [V][6] as met2_t2_fit's columns; est_signal [V][nTE]; sse [V]; iters [V] int32; status [V].
 * V = 0 is a no-op; bad arguments (sizes, NULL pointers, an empty box, V >= 2^31) return MET2_ERR_ARG before anything
 * is enqueued. */
typedef struct met2_param_cfg {
    int32_t nTE, nT2;
    int32_t max_iter;         /* Levenberg-Marquardt iterations (2000); MET2_ST_ITMAX when reached */
    int32_t reserved;
    double tau, TR, T1;       /* ms: echo spacing, repetition time, T1 of the dictionary */
    double t2_lo[3], t2_hi[3];/* ms: T2 box of the myelin, intra/extra-cellular and free-water pools */
    double fa_lo, fa_hi;      /* deg: flip-angle box (90, 180) */
    double mu0, mu_max;       /* initial damping (1e-3) and the cap that stops the iteration (1e16) */
    double ftol, xtol;        /* relative decrease of the cost (1e-12), scaled step (1e-10) */
} met2_param_cfg;
int met2_param_fit(const double* sig, const double* fa_deg, const double* fsol, const uint32_t* status_in, int64_t V,
                   const met2_param_cfg* cfg, const double* logT2, const uint8_t* comp, double* params, double* maps,
                   double* est_signal, double* sse, int32_t* iters, uint32_t* status, void* stream);

/* Rician-likelihood spectrum fitting (no counterpart in the reference): majorize-minimize iterations of warm-started
 * Tikhonov NNLS solves with modified data yt = y * I1/I0(y f / sn^2), started from the point fit.  Definition in
 * csrc/met2_rician.cu; the NumPy restatement is tests/rician_oracle.py.
 * Inputs are the point fit's: sig [V][nTE] raw signals, fa_index [V], lam [V] (any lam >= 0; the pipeline passes reg
 * under MET2_T2_FLAG_REG_IS_LAMBDA), x0 [V][nT2] = fsol / sig[0] and status_in [V]; sigma [V] is the noise SD in raw
 * signal units.  G, dicT, kband as for met2_t2_fit.  Outputs: x [V][nT2] (normalised spectra; met2_spatial_finish turns
 * them into fsol / est_signal / maps), iters [V] int32 (MM solves run), status [V] = status_in plus MET2_ST_MM_CAP,
 * MET2_ST_ITMAX and MET2_ST_BAD_SIGMA | MET2_ST_SKIPPED.  sigma = 0 reproduces the point fit (iters 0, x = x0).
 * Gram-domain sizes (nT2 <= 128, nTE <= 64), V < 2^31, max_iter >= 1, tol finite and >= 0; V = 0 is a no-op; bad
 * arguments return MET2_ERR_ARG before anything is enqueued.
 * met2_bessel_ratio writes A(z) = I1(z) / I0(z) of the kernel's routine for n HOST values z to out (host memory) and
 * returns n (MET2_ERR_ARG for n < 0 or a NULL pointer with n > 0). */
int met2_rician_fit(const double* sig, const int32_t* fa_index, const double* lam, const double* sigma,
                    const double* x0, const uint32_t* status_in, int64_t V, int nTE, int nT2, int nA, const double* G,
                    const double* dicT, const double* kband, int max_iter, double tol, double* x, int32_t* iters,
                    uint32_t* status, void* stream);
int64_t met2_bessel_ratio(const double* z, int64_t n, double* out);

/* Diagnostics */
const char* met2_last_error(void);
int met2_version(void);
/* MET2_ECHO_RANK (small = 0) or MET2_ECHO_RANK_SMALL (small != 0) of this library: the values of R that
 * met2_echo_basis / met2_t2_cfg.echo_rank accept for met2_t2_fit_echo. */
int met2_echo_rank(int small);
/* number of kernel launches enqueued by this library in this process so far (for bench.py's gpu_launches) */
int64_t met2_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* MET2_H_ */
