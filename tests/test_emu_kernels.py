"""The T2 fit kernels' OWN SOURCE (csrc/met2_t2_impl.cuh, met2_nnls.cuh, met2_t2_echo.cu) compiled by g++ against the
single-threaded SIMT emulator of tests/emu and run on the CPU — control flow, shared-memory indexing, warp collectives
and the blocked FP64-MMA factorisation included — against voxels fitted by the unmodified reference
(tests/golden/config2_subset.npz) and against the oracle.  This container has no GPU; the `-m gpu` tests repeat the same
comparisons on the device.  Tolerances are BASELINE.json's: active sets bit-exact, spectra 1e-6 relative, maps 1e-4.

Every kernel is run under three lane-scheduling orders (0..31, 31..0, a fresh random permutation every round): a result
that depends on the order means a missing barrier between a write and a read of two lanes.
"""
import os

import numpy as np
import pytest

import met2_oracle as O
from emu import emu

ORDERS = ("forward", "reverse", "shuffle")


@pytest.fixture(scope="module")
def setup(golden_config2):
    gr = O._grids("X2", "I", "spline", 40.0, 32, 10.0, 1000.0)
    Dic = O.create_Dic_3D(60, gr["T2s"], gr["T1s"], 32, 10.0, gr["alpha_values"], 1000.0)
    emu.build()
    return dict(gr=gr, Dic=Dic, g=golden_config2)


def _run(order, sig, fa, Dic, *args, **kw):
    """met2_t2_fit under the emulator with the given lane-scheduling order.  The dictionary is cut down to the flip
    angles these voxels use (the shared factor tables are built per angle: 273 angles would only cost emulation time);
    an out-of-range index stays out of range."""
    fa = np.asarray(fa)
    valid = (fa >= 0) & (fa < Dic.shape[2])
    uniq, inv = np.unique(fa[valid], return_inverse=True)
    fa_c = np.full(fa.shape, len(uniq) + 5, dtype=np.int32)
    fa_c[valid] = inv
    old = os.environ.get("SIMT_EMU_ORDER")
    os.environ["SIMT_EMU_ORDER"] = order
    try:
        return emu.t2_fit(sig, fa_c, np.ascontiguousarray(Dic[:, :, uniq]), *args, **kw)
    finally:
        if old is None:
            del os.environ["SIMT_EMU_ORDER"]
        else:
            os.environ["SIMT_EMU_ORDER"] = old


def _pick(g, n, offset=0):
    sel = np.arange(offset, len(g["sig"]), len(g["sig"]) // n)[:n]
    return sel, g["sig"][sel], g["fa_idx"][sel].astype(np.int32)


def _check(out, f_ref, reg_ref, ind_m, tol_f=1e-6):
    assert np.all(out["status"] == 0)
    assert np.array_equal(out["fsol"] > 0, f_ref > 0)                                  # active sets bit-exact
    scale = np.abs(f_ref).max(axis=1, keepdims=True)
    assert np.max(np.abs(out["fsol"] - f_ref) / scale) < tol_f
    assert np.max(np.abs(out["reg"] - reg_ref) / np.abs(reg_ref)) < 1e-6
    mwf = f_ref[:, ind_m].sum(1) / f_ref.sum(1)
    assert np.max(np.abs(out["maps"][:, 0] - mwf)) < 1e-4


def _same(a, b):
    return all(np.array_equal(a[k], b[k]) for k in ("fsol", "est_signal", "reg", "maps", "status"))


def test_production_x2_kernel_against_reference(setup):
    """t2_fit_kernel<2,1,X2> (warm starts, full-set start, Brent-best snapshot) vs the unmodified reference."""
    g, gr = setup["g"], setup["gr"]
    sel, sig, fa = _pick(g, 10)
    out = _run("forward", sig, fa, setup["Dic"], gr["L"], gr["T2s"], "X2", flags=16)
    _check(out, g["f"][sel], g["reg"][sel], gr["ind_m"])
    for o in ORDERS[1:]:                                     # lane-order invariance on the first voxels
        other = _run(o, sig[:4], fa[:4], setup["Dic"], gr["L"], gr["T2s"], "X2", flags=16)
        assert all(np.array_equal(out[k][:4], other[k]) for k in ("fsol", "est_signal", "reg", "maps", "status"))
    cold = _run("forward", sig[:4], fa[:4], setup["Dic"], gr["L"], gr["T2s"], "X2", flags=4)   # MET2_T2_FLAG_COLD_START
    _check(cold, g["f"][sel[:4]], g["reg"][sel[:4]], gr["ind_m"])


def test_echo_space_x2_kernel_against_reference(setup):
    """The experimental echo-space kernel (met2_t2_echo.cu): same tolerances, both starting strategies."""
    g, gr = setup["g"], setup["gr"]
    sel, sig, fa = _pick(g, 10, offset=7)
    outs = [_run("forward", sig, fa, setup["Dic"], gr["L"], gr["T2s"], "X2", flags=16, echo=True)]
    _check(outs[0], g["f"][sel], g["reg"][sel], gr["ind_m"], tol_f=1e-8)
    for o in ORDERS[1:]:
        other = _run(o, sig[:4], fa[:4], setup["Dic"], gr["L"], gr["T2s"], "X2", flags=16, echo=True)
        assert all(np.array_equal(outs[0][k][:4], other[k]) for k in ("fsol", "est_signal", "reg", "maps", "status"))
    # est_signal = D f * km (motor...:155) and the lambda-returning variant
    D = np.transpose(setup["Dic"], (2, 0, 1))[fa]
    assert np.allclose(outs[0]["est_signal"], np.einsum("vec,vc->ve", D, outs[0]["fsol"]), rtol=1e-10, atol=1e-9)
    nofull = _run("forward", sig[:6], fa[:6], setup["Dic"], gr["L"], gr["T2s"], "X2", flags=0, echo=True)
    _check(nofull, g["f"][sel[:6]], g["reg"][sel[:6]], gr["ind_m"], tol_f=1e-8)
    # rank 16 of the reduced space (what the plan picks for this protocol, batched.ECHO_TAIL_MAX): same active sets,
    # spectra in the accuracy class of the Gram-domain kernel
    r16 = _run("forward", sig[:6], fa[:6], setup["Dic"], gr["L"], gr["T2s"], "X2", flags=16, echo=True, echo_rank=16)
    _check(r16, g["f"][sel[:6]], g["reg"][sel[:6]], gr["ind_m"], tol_f=1e-7)
    lam = _run("forward", sig[:3], fa[:3], setup["Dic"], gr["L"], gr["T2s"], "X2", flags=16 | 1, echo=True)
    for i in range(3):
        Dv = np.ascontiguousarray(setup["Dic"][:, :, fa[i]])
        _, reg, _ = O.nnls_x2(Dv, sig[i] / sig[i, 0], gr["L"], 1.02)
        assert abs(lam["reg"][i] - reg) < 1e-9 * max(1.0, abs(reg))


def test_echo_space_without_tables_rejected_before_any_launch(setup):
    """MET2_T2_FLAG_ECHO_SPACE with NULL red_basis / red_coef is an argument error, returned before the sort kernels or
    anything else is enqueued."""
    g, gr = setup["g"], setup["gr"]
    _, sig, fa = _pick(g, 4)
    before = emu.lib().met2_launch_count()
    with pytest.raises(RuntimeError, match=r"\(-1\): met2_t2_fit: MET2_T2_FLAG_ECHO_SPACE needs the reduced echo basis"):
        _run("forward", sig, fa, setup["Dic"], gr["L"], gr["T2s"], "X2", flags=64)   # flag set, echo=False: no tables
    assert emu.lib().met2_launch_count() == before


def test_echo_space_invt2_and_rejects_non_diagonal(setup):
    g = setup["g"]
    gi = O._grids("X2", "InvT2", "spline", 40.0, 32, 10.0, 1000.0)
    sel, sig, fa = _pick(g, 8, offset=3)
    out = _run("shuffle", sig, fa, setup["Dic"], gi["L"], gi["T2s"], "X2", flags=0, echo=True)
    ref = [O.t2_fit_voxel(sig[i], np.ascontiguousarray(setup["Dic"][:, :, fa[i]]), "X2", gi["L"], gi["lambda_reg"])
           for i in range(len(sel))]
    _check(out, np.array([r[0] for r in ref]), np.array([r[2] for r in ref]), gi["ind_m"])
    prod = _run("forward", sig, fa, setup["Dic"], gi["L"], gi["T2s"], "X2", flags=0)
    assert np.array_equal(prod["fsol"] > 0, out["fsol"] > 0)
    # L2 is tridiagonal: the echo-space formulation does not apply -> every voxel skipped with MET2_ST_ECHO_BAD_L
    g2 = O._grids("X2", "L2", "spline", 40.0, 32, 10.0, 1000.0)
    bad = _run("forward", sig[:2], fa[:2], setup["Dic"], g2["L"], g2["T2s"], "X2", flags=0, echo=True)
    assert np.all(bad["status"] == (1 | 32)) and not bad["fsol"].any() and not bad["est_signal"].any()


def test_echo_space_lcurve_and_bayesreg_against_oracle(setup):
    """t2_echo_reg_kernel (met2_t2_echo_reg_impl.cuh): L-curve (algorithms.py:88-113) and BayesReg
    (bayesian_interpolation.py:84-126, evidence by the structured Cholesky sweep) in the reduced echo space, both ranks,
    I and InvT2, against the oracle: active sets bit-exact, the L-curve corner identical, BayesReg's lambda within the
    reproducibility of its flat evidence (InvT2: DESIGN.md §5)."""
    g, gr = setup["g"], setup["gr"]
    sel, sig, fa = _pick(g, 3, offset=5)
    Dv = [np.ascontiguousarray(setup["Dic"][:, :, a]) for a in fa]
    for method, rm, rank, tol_f, tol_reg in (("L_curve", "I", 16, 1e-8, 1e-12), ("L_curve", "InvT2", 24, 1e-8, 1e-12),
                                             ("BayesReg", "I", 16, 1e-7, 1e-6), ("BayesReg", "InvT2", 24, 1e-6, 1e-6)):
        grm = O._grids(method, rm, "spline", 40.0, 32, 10.0, 1000.0)
        out = _run("shuffle", sig, fa, setup["Dic"], grm["L"], gr["T2s"], method, echo=True, echo_rank=rank,
                   lambdas=gr["lambda_reg"])
        if rank == 16:       # lane-order invariance: a missing barrier between lanes shows up as a difference
            again = _run("reverse", sig, fa, setup["Dic"], grm["L"], gr["T2s"], method, echo=True, echo_rank=rank,
                         lambdas=gr["lambda_reg"])
            assert _same(out, again)
        for i in range(len(sel)):
            f_ref, s_ref, reg_ref = O.t2_fit_voxel(sig[i], Dv[i], method, grm["L"], gr["lambda_reg"])
            assert out["status"][i] == 0 and np.array_equal(out["fsol"][i] > 0, f_ref > 0), (method, rm, i)
            assert np.max(np.abs(out["fsol"][i] - f_ref)) < tol_f * np.abs(f_ref).max(), (method, rm, i)
            assert np.max(np.abs(out["est_signal"][i] - s_ref)) < 1e-6 * np.abs(s_ref).max()
            assert abs(out["reg"][i] - reg_ref) <= tol_reg * max(1.0, abs(reg_ref)), (method, rm, i)
    # L-curve with the Gram-domain / echo-space switch moved above the grid (MET2_LCURVE_SWITCH): every point is tried
    # in the Gram domain until the 32-position factor is full, which sends the rest of the grid to echo space — the
    # fall-back path of the driver; and with the switch at 0: the whole grid in echo space
    grm = O._grids("L_curve", "I", "spline", 40.0, 32, 10.0, 1000.0)
    for sw in ("100", "0"):
        os.environ["MET2_LCURVE_SWITCH"] = sw
        try:
            out = _run("forward", sig[:2], fa[:2], setup["Dic"], grm["L"], gr["T2s"], "L_curve", echo=True, echo_rank=16,
                       lambdas=gr["lambda_reg"])
        finally:
            del os.environ["MET2_LCURVE_SWITCH"]
        for i in range(2):
            f_ref, _, reg_ref = O.t2_fit_voxel(sig[i], Dv[i], "L_curve", grm["L"], gr["lambda_reg"])
            assert out["status"][i] == 0 and np.array_equal(out["fsol"][i] > 0, f_ref > 0), (sw, i)
            assert np.max(np.abs(out["fsol"][i] - f_ref)) < 1e-8 * np.abs(f_ref).max(), (sw, i)
            assert out["reg"][i] == reg_ref, (sw, i)


def test_edge_voxels_both_kernels(setup):
    """Empty / NaN / M[0] = 0 voxels and a bad FA index: flagged, all-zero outputs, neighbours unaffected
    (motor...:124-131, algorithms.py:56)."""
    g, gr = setup["g"], setup["gr"]
    sel, sig, fa = _pick(g, 6, offset=11)
    sig = sig.copy()
    fa = fa.copy()
    sig[1] = 0.0
    sig[2, 5] = np.nan
    sig[3, 0] = 0.0
    fa[4] = 999
    for echo in (False, True):
        out = _run("forward", sig, fa, setup["Dic"], gr["L"], gr["T2s"], "X2", flags=16, echo=echo)
        assert list(out["status"]) == [0, 1, 3, 1, 1, 0]
        assert not out["fsol"][1:5].any() and not out["est_signal"][1:5].any() and not out["reg"][1:5].any()
        keep = [0, 5]
        assert np.array_equal(out["fsol"][keep] > 0, g["f"][sel[keep]] > 0)
        assert np.max(np.abs(out["fsol"][keep] - g["f"][sel[keep]])) < 1e-6 * np.abs(g["f"][sel[keep]]).max()


def test_production_other_methods_against_oracle(setup):
    """NNLS (with its D-space refinement step), fixed-lambda Tikhonov (L = I and L2) and the L-curve grid + corner."""
    g, gr = setup["g"], setup["gr"]
    sel, sig, fa = _pick(g, 5, offset=19)
    Dv = [np.ascontiguousarray(setup["Dic"][:, :, a]) for a in fa]
    g2 = O._grids("X2", "L2", "spline", 40.0, 32, 10.0, 1000.0)
    cases = (("NNLS", gr["L"], {}), ("T2SPARC", gr["L"], {}), ("T2SPARC", g2["L"], {}),
             ("L_curve", gr["L"], dict(lambdas=gr["lambda_reg"])))
    for method, L, kw in cases:
        out = _run("shuffle", sig, fa, setup["Dic"], L, gr["T2s"], method, **kw)
        for i in range(len(sel)):
            f_ref, s_ref, reg_ref = O.t2_fit_voxel(sig[i], Dv[i], method, L, gr["lambda_reg"])
            assert out["status"][i] == 0
            assert np.array_equal(out["fsol"][i] > 0, f_ref > 0), (method, i)
            assert np.max(np.abs(out["fsol"][i] - f_ref)) < 1e-6 * np.abs(f_ref).max(), (method, i)
            assert np.max(np.abs(out["est_signal"][i] - s_ref)) < 1e-6 * np.abs(s_ref).max()
            assert abs(out["reg"][i] - reg_ref) <= 1e-9 * max(1.0, abs(reg_ref))


def test_production_bayesreg_and_gcv_against_oracle(setup):
    """BayesReg (evidence with the blocked n x n factorisation, erf, log-det; bayesian_interpolation.py:84-126): lambda
    and spectrum against the oracle.  GCV (algorithms.py:276-296): the criterion is not reproducible to better than
    ~1e-3 in lambda even by the reference itself (DESIGN.md §5), so the bar is the derived map, |dMWF| < 1e-4.
    Both under the shuffled lane order; the GCV kernel's pivoted-Cholesky loop exit used to be a write-after-read race
    between lanes that only this emulator's sequential schedule exposed."""
    g, gr = setup["g"], setup["gr"]
    sel, sig, fa = _pick(g, 3, offset=5)
    Dv = [np.ascontiguousarray(setup["Dic"][:, :, a]) for a in fa]
    out = _run("shuffle", sig, fa, setup["Dic"], gr["L"], gr["T2s"], "BayesReg")
    again = _run("reverse", sig, fa, setup["Dic"], gr["L"], gr["T2s"], "BayesReg")
    assert _same(out, again)
    for i in range(len(sel)):
        f_ref, _, reg_ref = O.t2_fit_voxel(sig[i], Dv[i], "BayesReg", gr["L"], gr["lambda_reg"])
        assert out["status"][i] == 0 and np.array_equal(out["fsol"][i] > 0, f_ref > 0)
        assert np.max(np.abs(out["fsol"][i] - f_ref)) < 1e-6 * np.abs(f_ref).max()
        assert abs(out["reg"][i] - reg_ref) < 1e-6 * abs(reg_ref)
    out = _run("shuffle", sig, fa, setup["Dic"], gr["L"], gr["T2s"], "GCV")
    again = _run("forward", sig, fa, setup["Dic"], gr["L"], gr["T2s"], "GCV")
    assert _same(out, again)
    for i in range(len(sel)):
        f_ref, _, _ = O.t2_fit_voxel(sig[i], Dv[i], "GCV", gr["L"], gr["lambda_reg"])
        assert out["status"][i] == 0
        assert abs(out["maps"][i, 0] - f_ref[gr["ind_m"]].sum() / f_ref.sum()) < 1e-4


def test_fa_stage_kernels_against_reference(setup):
    """csrc/met2_fa.cu under the emulator: fa_search_kernel (warm-started plain NNLS per search angle) ->
    spline_weights_kernel -> fa_select_kernel (not-a-knot spline + the bounded-Brent replica + grid snap, NNLS at the
    chosen angle) -> reduce_partials_kernel.  Spline method against the FA indices / km the unmodified reference
    produced (fa_estimation.py:35-72); brute force against the oracle (fa_estimation.py:74-112).  Bit-exact indices."""
    g, gr = setup["g"], setup["gr"]
    sel = np.arange(3, len(g["sig"]), len(g["sig"]) // 8)[:8]
    sig = g["sig"][sel]
    DicLR = O.create_Dic_3D(60, gr["T2s"], gr["T1s"], 32, 10.0, gr["alpha_spline"], 1000.0)
    outs = []
    for order in ORDERS:
        os.environ["SIMT_EMU_ORDER"] = order
        try:
            outs.append(emu.fa_fit(sig, setup["Dic"], gr["alpha_values"], DicLR, gr["alpha_spline"]))
        finally:
            del os.environ["SIMT_EMU_ORDER"]
    out = outs[0]
    assert np.all(out["status"] == 0)
    assert np.array_equal(out["fa_index"], g["fa_idx"][sel])
    assert np.array_equal(out["fa_deg"], gr["alpha_values"][g["fa_idx"][sel]])
    assert np.max(np.abs(out["km"] - g["km"][sel]) / g["km"][sel]) < 1e-9
    for other in outs[1:]:
        assert all(np.array_equal(out[k], other[k]) for k in ("fa_index", "fa_deg", "km", "status"))
        assert np.allclose(out["fsol_sum"], other["fsol_sum"], rtol=1e-13, atol=0)   # summation order follows the warps
    # the search has two kernels: thread per voxel (default) and warp per voxel, which also redoes the voxels the first one
    # hands back (positive set above its cap: forced here with a cap of 3 columns).  Same indices on every path.
    for env in ({"MET2_FA_SEARCH": "warp"}, {"MET2_FA_THREAD_PCAP": "3"}):
        os.environ.update(env)
        try:
            alt = emu.fa_fit(sig, setup["Dic"], gr["alpha_values"], DicLR, gr["alpha_spline"])
        finally:
            for k in env:
                del os.environ[k]
        assert all(np.array_equal(out[k], alt[k]) for k in ("fa_index", "fa_deg", "status")), env
        assert np.max(np.abs(out["km"] - alt["km"]) / out["km"]) < 1e-12
    a91 = np.linspace(90.0, 180.0, 91)
    D91 = O.create_Dic_3D(60, gr["T2s"], gr["T1s"], 32, 10.0, a91, 1000.0)
    sig_b = sig[:5].copy()
    sig_b[3] = 0.0                                                  # empty voxel: index 0, status skipped
    out = emu.fa_fit(sig_b, D91, a91)
    FA, idx, KM, F = O.fitting_slice_FA_brute_force((sig_b.sum(1) > 0).astype(float), sig_b, 5, D91, a91)
    assert list(out["status"]) == [0, 0, 0, 1, 0]
    assert np.array_equal(out["fa_index"], idx.astype(np.int32)) and np.array_equal(out["fa_deg"], FA)
    assert np.max(np.abs(out["km"] - KM)) < 1e-8 * KM.max()
    assert np.max(np.abs(out["fsol_sum"] - F)) < 1e-6 * np.abs(F).max()
    os.environ["MET2_FA_THREAD_PCAP"] = "3"
    try:
        alt = emu.fa_fit(sig_b, D91, a91)
    finally:
        del os.environ["MET2_FA_THREAD_PCAP"]
    assert all(np.array_equal(out[k], alt[k]) for k in ("fa_index", "fa_deg", "status"))


def _synthetic(npc, nte, nv, method, matrix, seed=3):
    """Three-compartment spectra (myelin 20 ms, IE 60-90 ms, free water 1.5 s) through the oracle's EPG dictionary."""
    gr = O._grids(method, matrix, "brute-force", 40.0, nte, 10.0, 1000.0, npc=npc, n_alphas=7)
    Dic = O.create_Dic_3D(npc, gr["T2s"], gr["T1s"], nte, 10.0, gr["alpha_values"], 1000.0)
    rng = np.random.default_rng(seed)
    fa = rng.integers(0, 7, nv).astype(np.int32)
    lt = np.log(gr["T2s"])
    sig = np.zeros((nv, nte))
    for i in range(nv):
        spec = (0.15 * np.exp(-0.5 * ((lt - np.log(20.0)) / 0.15) ** 2)
                + 0.8 * np.exp(-0.5 * ((lt - np.log(rng.uniform(60.0, 90.0))) / 0.12) ** 2)
                + 0.05 * np.exp(-0.5 * ((lt - np.log(1500.0)) / 0.1) ** 2))
        s = Dic[:, :, fa[i]] @ spec
        sig[i] = 1000.0 * np.abs(s + rng.normal(0.0, s[0] / 150.0, nte))
    return gr, Dic, sig, fa


@pytest.mark.parametrize("method,matrix,npc,nte,nv,tol,echo", [
    ("T2SPARC", "InvT2", 96, 32, 1, 1e-6, False),    # the reference's T2SPARC grid in the Gram domain: three column slots
                                                     # per lane (one voxel: 28 s each under emulation; the echo-space
                                                     # kernel that runs by default has its own test)
    ("NNLS", "I", 100, 48, 3, 1e-6, False),          # BASELINE.json config 4 sizes: four column slots, two echo slots
    ("X2", "I", 100, 48, 2, 1e-6, False),
    ("BayesReg", "InvT2", 100, 48, 2, 1e-3, False),  # flat evidence: the reference does not reproduce itself (DESIGN.md §5)
    ("BayesReg", "InvT2", 100, 48, 2, 1e-3, True),   # config 4 in the reduced echo space (t2_echo_reg_kernel<5, 4, 2>)
    ("L_curve", "I", 100, 48, 2, 1e-6, True),
])
def test_production_kernels_large_sizes(method, matrix, npc, nte, nv, tol, echo):
    emu.build()
    gr, Dic, sig, fa = _synthetic(npc, nte, nv, method, matrix)
    out = _run("shuffle", sig, fa, Dic, gr["L"], gr["T2s"], method, lambdas=gr["lambda_reg"], echo=echo)
    assert np.all(out["status"] == 0)
    for i in range(nv):
        f_ref, s_ref, reg_ref = O.t2_fit_voxel(sig[i], np.ascontiguousarray(Dic[:, :, fa[i]]), method, gr["L"],
                                               gr["lambda_reg"])
        assert np.array_equal(out["fsol"][i] > 0, f_ref > 0)
        assert np.max(np.abs(out["fsol"][i] - f_ref)) < tol * np.abs(f_ref).max()
        assert abs(out["reg"][i] - reg_ref) <= tol * max(1.0, abs(reg_ref))
        assert abs(out["maps"][i, 0] - f_ref[gr["ind_m"]].sum() / f_ref.sum()) < 1e-4


def test_whole_chain_against_the_reference_orchestrator_run():
    """Every kernel of the path in sequence, emulated: EPG dictionary -> NESMA -> Gaussian smoothing -> FA spline search ->
    X2-I fit + maps, against the output volumes of the UNMODIFIED reference's motor_recon_met2 run end to end
    (tests/golden/pipeline_nesma_x2.npz, oracle/make_golden_pipeline.py; denoise=NESMA, FA_smooth=yes).  The two
    preprocessing stages run on the whole 14x12x10 volume, the fits on every 19th masked voxel."""
    g = dict(np.load(os.path.join(os.path.dirname(__file__), "golden", "pipeline_nesma_x2.npz")))
    mask = g["mask"].astype(np.int64)
    data = g["data"] * mask[..., None]
    data[data < 0.0] = 0.0                                                     # motor...:178-180
    gr = O._grids("X2", "I", "spline", 40.0, 32, float(g["TE"][1] - g["TE"][0]), 1000.0)
    tau = float(g["TE"][1] - g["TE"][0])
    dic, _ = emu.epg_dictionary(gr["alpha_values"], gr["T2s"], gr["T1s"], 32, tau, 1000.0)
    dic_lr, _ = emu.epg_dictionary(gr["alpha_spline"], gr["T2s"], gr["T1s"], 32, tau, 1000.0)
    Dic, DicLR = np.transpose(dic, (1, 2, 0)), np.transpose(dic_lr, (1, 2, 0))
    den = emu.nesma_filter(data, mask.astype(np.int32))                        # Step 1 (motor...:305-333)
    smooth = emu.gaussian_smooth(den, 2.0)                                     # FA-stage copy (motor...:336-346)
    flat = np.nonzero(mask.reshape(-1) > 0)[0][::19]
    assert len(flat) >= 30
    sig = den.reshape(-1, 32)[flat]
    sig_fa = smooth.reshape(-1, 32)[flat]
    fa = emu.fa_fit(sig_fa, Dic, gr["alpha_values"], DicLR, gr["alpha_spline"])          # Step 2
    assert np.array_equal(fa["fa_deg"], g["FA"].reshape(-1)[flat])                      # FA map bit-exact
    out = _run("shuffle", sig, fa["fa_index"], Dic, gr["L"], gr["T2s"], "X2", flags=16)  # Steps 3 and 4
    f_ref = g["fsol_4D"].reshape(-1, 60)[flat]
    assert np.array_equal(out["fsol"] > 0, f_ref > 0)                                    # active sets bit-exact
    scale = np.abs(f_ref).max(axis=1, keepdims=True)
    scale[scale == 0] = 1.0
    assert np.max(np.abs(out["fsol"] - f_ref) / scale) < 1e-6
    for i, k in enumerate(("MWF", "IEWF", "FWF", "T2_M", "T2_IE")):
        assert np.max(np.abs(out["maps"][:, i] - g[k].reshape(-1)[flat])) < 1e-4, k
    for got, k in ((out["maps"][:, 5], "TWC"), (out["reg"], "reg_param")):
        ref = g[k].reshape(-1)[flat]
        assert np.max(np.abs(got - ref)) <= 1e-6 * np.abs(ref).max(), k
    s_ref = g["Est_Signal"].reshape(-1, 32)[flat]
    assert np.max(np.abs(out["est_signal"] - s_ref)) <= 1e-6 * np.abs(s_ref).max()


def test_echo_basis_kernel():
    """met2_echo_basis (column-pivoted Gram-Schmidt per angle): U orthonormal (directions below the rounding of D are
    zero vectors), U C = D to rounding, residual reported per angle — 32 x 60 and the config-4 shape 48 x 100."""
    for npc, nte, tau in ((60, 32, 10.0), (100, 48, 8.0)):
        T2s = np.logspace(1, np.log10(2000.0), npc)
        Dic = O.create_Dic_3D(npc, T2s, 1000.0 * np.ones(npc), nte, tau, np.array([91.0, 133.0, 180.0]), 1000.0)
        dic = np.ascontiguousarray(np.transpose(Dic, (2, 0, 1)))
        U, C, tail = emu.echo_basis(dic)
        assert tail.max() <= 1e-15
        for a in range(3):
            UtU = U[a].T @ U[a]
            nz = np.diag(UtU) > 0.5
            assert np.abs(UtU - np.diag(nz.astype(float))).max() < 1e-14
            assert np.abs(U[a] @ C[a].T - dic[a]).max() <= 2e-15 * np.abs(dic[a]).max()
        # rank 16 (MET2_ECHO_RANK_SMALL): the measured residual decides — the 32-echo protocol is inside the 4e-12 bound of
        # batched.ECHO_TAIL_MAX (and far above the rank-24 bound, so the two ranks cannot be confused), the 48-echo one is not
        U16, C16, tail16 = emu.echo_basis(dic, 16)
        for a in range(3):
            resid = np.abs(U16[a] @ C16[a].T - dic[a]).max() / np.abs(dic[a]).max()
            assert resid <= 4.0 * tail16[a] + 1e-15            # the kernel's own measure is honest
        if nte == 32:
            assert 1e-14 < tail16.max() <= 4e-12, tail16
        else:
            assert tail16.max() > 4e-12, tail16
    few = emu.echo_basis(np.random.default_rng(0).uniform(size=(1, 8, 12)))      # fewer echoes than R: zero directions
    assert np.abs(few[0][0] @ few[1][0].T - np.random.default_rng(0).uniform(size=(1, 8, 12))[0]).max() < 1e-14
    assert few[2][0] <= 1e-15
    full = emu.echo_basis(np.random.default_rng(1).uniform(size=(1, 32, 60)))    # full-rank dictionary: reported, not hidden
    assert full[2][0] > 1e-3


@pytest.mark.parametrize("matrix,npc,nte", [("InvT2", 96, 32), ("I", 96, 32), ("InvT2", 60, 32), ("InvT2", 100, 48)])
def test_echo_space_fixed_lambda_kernel(matrix, npc, nte):
    """t2_echo_tik_kernel (T2SPARC in the reduced echo space): one solve per voxel from the empty set with rank-one
    updates of the 24 x 24 factor only; the reference's 96-bin grid uses three column slots per lane; 48 echoes / 100
    bins (config-4 sizes): four column slots, two echo slots."""
    emu.build()
    gr, Dic, sig, fa = _synthetic(npc, nte, 6 if nte == 32 else 3, "T2SPARC", matrix)
    outs = [_run(o, sig, fa, Dic, gr["L"], gr["T2s"], "T2SPARC", echo=True) for o in ORDERS]
    assert _same(outs[0], outs[1]) and _same(outs[0], outs[2])
    out = outs[0]
    assert np.all(out["status"] == 0) and np.all(out["reg"] == 1.8)
    for i in range(len(sig)):
        f_ref, s_ref, _ = O.t2_fit_voxel(sig[i], np.ascontiguousarray(Dic[:, :, fa[i]]), "T2SPARC", gr["L"],
                                         gr["lambda_reg"])
        assert np.array_equal(out["fsol"][i] > 0, f_ref > 0)
        assert np.max(np.abs(out["fsol"][i] - f_ref)) < 1e-8 * np.abs(f_ref).max()
        assert np.max(np.abs(out["est_signal"][i] - s_ref)) < 1e-8 * np.abs(s_ref).max()
        assert abs(out["maps"][i, 0] - f_ref[gr["ind_m"]].sum() / f_ref.sum()) < 1e-8


def test_gcv_objective_and_grid_modes(setup):
    """The GCV kernel's objective (algorithms.py:285-296, quirks included) at fixed lambdas (MET2_T2_FLAG_GCV_EVAL) and
    its lambda-grid mode (MET2_T2_FLAG_GCV_GRID, BASELINE.json configs[2]) against the oracle.  The criterion sits on
    a truncated pseudo-inverse whose cut-off is at rounding level for some eigenvalues (SURVEY.md a-8), so the
    objective is compared statistically like in the GPU test."""
    g, gr = setup["g"], setup["gr"]
    sel, sig, fa = _pick(g, 8, offset=13)
    Dv = [np.ascontiguousarray(setup["Dic"][:, :, a]) for a in fa]
    d = []
    for lam in (1e-3, 0.1, 3.8197):
        out = _run("shuffle", sig, fa, setup["Dic"], gr["L"], gr["T2s"], "GCV", flags=8, lambda_fixed=lam)
        assert not (out["status"] & 0xffff).any()
        kept = (out["status"].astype(np.int64) >> 16) & 0xff      # rank of the truncated pseudo-inverse (met2.h)
        for i in range(len(sel)):
            M = sig[i] / sig[i, 0]
            with np.errstate(all="ignore"):
                ref = O.obj_nnls_gcv(lam, Dv[i], gr["L"], np.concatenate((M, np.zeros(60))), 32, np.eye(32))
                f, _ = O.nnls(np.concatenate((Dv[i], np.sqrt(lam) * gr["L"])), np.concatenate((M, np.zeros(60))))
                s = f > 0
                Dr, Lr = Dv[i][:, s], gr["L"][s, s]
                rank = np.linalg.lstsq(Dr.T @ Dr + lam * (Lr.T @ Lr), Dr.T, rcond=None)[2]
            assert kept[i] == rank, (lam, i, kept[i], rank)
            d.append(abs(out["reg"][i] - ref))
    d = np.array(d)
    assert np.median(d) < 1e-4 and (d < 1e-2).mean() > 0.9, (np.median(d), d.max())
    lams = np.ascontiguousarray(gr["lambda_reg"][1:])
    out = _run("forward", sig, fa, setup["Dic"], gr["L"], gr["T2s"], "GCV", flags=32, lambdas=lams)
    assert not out["status"].any()
    gi = np.array([int(np.argmin(np.abs(np.log(lams) - np.log(l)))) for l in out["reg"]])
    assert np.allclose(lams[gi], out["reg"], rtol=1e-14)                      # a grid value was returned
    gi_ref = np.zeros(len(sel), dtype=int)
    for i in range(len(sel)):
        fr, reg, costs = O.nnls_gcv_grid(Dv[i], sig[i] / sig[i, 0], gr["L"], lams)
        gi_ref[i] = int(np.argmin(costs))
        if gi_ref[i] == gi[i]:
            assert np.array_equal(out["fsol"][i] > 0, fr > 0)
            assert np.max(np.abs(out["fsol"][i] - fr * sig[i, 0])) < 1e-6 * np.abs(fr * sig[i, 0]).max()
    assert (np.abs(gi - gi_ref) <= 1).mean() >= 0.75, (gi, gi_ref)


def test_odd_sizes_and_tile_scheduling():
    """Sizes off the beaten path through the real host code: 24 echoes, 50 bins (neither a multiple of 32 nor even rows
    of the Gram table), three flip angles, 301 voxels (ragged last tile, tiles of 32 forced through MET2_T2_TILE so that
    one flip angle spans several tiles), two emulated SMs pulling tiles from the shared counter."""
    emu.build()
    gr, Dic, sig, fa = _synthetic(50, 24, 301, "T2SPARC", "L1", seed=9)
    fa = (fa % 3).astype(np.int32)
    Dic = np.ascontiguousarray(Dic[:, :, :3])
    old = os.environ.get("MET2_T2_TILE")
    os.environ["MET2_T2_TILE"] = "32"
    try:
        outs = {m: emu.t2_fit(sig, fa, Dic, gr["L"], gr["T2s"], m, warps=3) for m in ("NNLS", "T2SPARC")}
    finally:
        if old is None:
            del os.environ["MET2_T2_TILE"]
        else:
            os.environ["MET2_T2_TILE"] = old
    for method, out in outs.items():
        assert not out["status"].any()
        for i in range(0, len(sig), 7):
            f_ref, s_ref, reg_ref = O.t2_fit_voxel(sig[i], np.ascontiguousarray(Dic[:, :, fa[i]]), method, gr["L"],
                                                   gr["lambda_reg"])
            assert np.array_equal(out["fsol"][i] > 0, f_ref > 0), (method, i)
            assert np.max(np.abs(out["fsol"][i] - f_ref)) < 1e-6 * np.abs(f_ref).max(), (method, i)
            assert np.max(np.abs(out["est_signal"][i] - s_ref)) < 1e-6 * np.abs(s_ref).max()
        # every voxel was fitted exactly once: no voxel left at its poison value, TWC > 0 everywhere
        assert np.isfinite(out["fsol"]).all() and (out["maps"][:, 5] > 0).all()


@pytest.mark.parametrize("npc", [96, 100])
def test_plain_nnls_wide_grids_against_reference(golden_plain_wide, npc):
    """Plain NNLS on the 96- / 100-bin grids, where long-T2 columns are nearly collinear and the Gram-domain dependence
    test rho^2 = G_jj - r.r loses its digits: with the D-space evaluation of nearly dependent candidates
    (dspace_candidate, met2_nnls.cuh) the production kernel lands on the reference's support (DESIGN.md §5; without it:
    1 disagreement in 1 500 voxels).  256 voxels here; all 20 480 in the -m gpu suite."""
    g = golden_plain_wide
    sel = np.arange(11, 20480, 80)[:256]
    sig, fa = g["sig"][sel], g["fa_idx"][sel]
    uniq, inv = np.unique(fa, return_inverse=True)
    T2s = np.logspace(1, np.log10(2000.0), npc)
    Dic = O.create_Dic_3D(npc, T2s, 1000.0 * np.ones(npc), 32, 10.0, np.linspace(90, 180, 273)[uniq], 1000.0)
    out = emu.t2_fit(sig, inv.astype(np.int32), Dic, np.eye(npc), T2s, "NNLS")
    f_ref = g["f%d" % npc][sel]
    assert np.all(out["status"] == 0)
    assert np.array_equal(out["fsol"] > 0, f_ref > 0)
    assert np.max(np.abs(out["fsol"] - f_ref) / np.abs(f_ref).max(axis=1, keepdims=True)) < 1e-6
