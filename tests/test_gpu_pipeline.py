"""The stage sequence and output tables of pipeline.py on one GPU: MultiGpuFit with bootstrap and the parametric fit
equals fit_voxels byte for byte (also with two plans sharing the device, so the voxel list is dealt to two "devices"),
the volumes recon_arrays returns for every valid option combination, and the buffers host_buffers allocates."""
import itertools

import numpy as np
import pytest
import torch

from multicomponent_t2_toolbox_b200 import batched, pipeline
from multicomponent_t2_toolbox_b200.phantom import make_phantom

pytestmark = pytest.mark.gpu

PER_VOXEL = ("fa_index", "fa_deg", "km", "fa_status", "fsol", "est_signal", "reg", "maps", "status", "boot_stats",
             "boot_n_valid", "param_params", "param_maps", "param_est_signal", "param_sse", "param_iters", "param_status")


def _plan():
    return batched.Met2Plan(32, 10.0, 1000.0, reg_method="X2", reg_matrix="I", FA_method="spline", device="cuda:0")


def test_multi_gpu_fit_with_bootstrap_and_parametric_equals_fit_voxels():
    ph = make_phantom((24, 20, 6), seed=12, fa_mode="b1")
    sig = np.ascontiguousarray(ph["data"].reshape(-1, 32))
    sig[5] = 0.0                                          # a skipped voxel
    plan = _plan()
    ref = pipeline.fit_voxels(plan, sig, n_bootstrap=4, parametric=True)
    assert set(ref) == set(PER_VOXEL) | {"fsol_sum"}
    assert ref["status"][5] & batched.ST_SKIPPED
    pin = torch.as_tensor(sig).pin_memory()
    for plans in ([plan], [plan, _plan()]):
        multi = pipeline.MultiGpuFit(plans, chunks_per_device=3)
        for rep in range(2):                              # the second call reuses the per-device buffers
            out = multi.fit(pin, n_bootstrap=4, parametric=True)
            for k in PER_VOXEL:
                assert out[k].dtype == ref[k].dtype and out[k].shape == ref[k].shape, (k, len(plans), rep)
                assert out[k].tobytes() == ref[k].tobytes(), (k, len(plans), rep)
            assert np.allclose(out["fsol_sum"], ref["fsol_sum"], rtol=1e-12, atol=0)


def _expected_volumes(shape, nt, npc, n_bootstrap, parametric, diagnostics, rois, fa_only):
    f64, i32 = np.dtype(np.float64), np.dtype(np.int32)
    vol = {"FA": (f64, shape), "FA_index": (f64, shape), "mean_T2_dist": (f64, (npc,)), "T2s": (f64, (npc,))}
    if diagnostics:
        vol["diagnostics"] = None
    if rois:
        vol["roi"] = None
    if fa_only:
        return vol
    vol.update({"MWF": (f64, shape), "IEWF": (f64, shape), "FWF": (f64, shape), "T2_M": (f64, shape),
                "T2_IE": (f64, shape), "TWC": (f64, shape), "reg_param": (f64, shape),
                "fsol_4D": (f64, shape + (npc,)), "Est_Signal": (f64, shape + (nt,)), "status": (i32, shape)})
    if n_bootstrap:
        vol.update({"MWF_bootstrap": (f64, shape + (4,)), "IEWF_bootstrap": (f64, shape + (4,)),
                    "FWF_bootstrap": (f64, shape + (4,)), "T2_M_bootstrap": (f64, shape + (4,)),
                    "T2_IE_bootstrap": (f64, shape + (4,)), "TWC_bootstrap": (f64, shape + (4,)),
                    "bootstrap_n_valid": (i32, shape)})
    if parametric:
        vol.update({"MWF_3pool": (f64, shape), "IEWF_3pool": (f64, shape), "FWF_3pool": (f64, shape),
                    "T2_M_3pool": (f64, shape), "T2_IE_3pool": (f64, shape), "T2_FW_3pool": (f64, shape),
                    "FA_3pool": (f64, shape), "TWC_3pool": (f64, shape), "SSE_3pool": (f64, shape),
                    "Est_Signal_3pool": (f64, shape + (nt,))})
    return vol


def test_recon_arrays_volumes_for_every_option_combination():
    ph = make_phantom((6, 5, 4), seed=9, fa_mode="b1", mask_mode="ellipsoid")
    shape, nt = ph["mask"].shape, ph["data"].shape[3]
    rois = (np.arange(ph["mask"].size) % 3).reshape(shape)
    plan = batched.Met2Plan(nt, ph["TE_array"][1] - ph["TE_array"][0], ph["TR"], reg_method="X2", reg_matrix="I",
                            FA_method="spline")
    for n_bootstrap, parametric, spatial_mu, diagnostics, with_rois, fa_only in itertools.product(
            (0, 4), (False, True), (0.0, 0.1), (False, True), (False, True), (False, True)):
        if spatial_mu > 0 and (n_bootstrap or parametric):
            continue
        opts = (n_bootstrap, parametric, spatial_mu, diagnostics, with_rois, fa_only)
        vol = pipeline.recon_arrays(ph["data"], ph["mask"], ph["TE_array"], ph["TR"], "X2", "I", "spline", plan=plan,
                                    n_bootstrap=n_bootstrap, parametric=parametric, spatial_mu=spatial_mu,
                                    spatial_sweeps=2, diagnostics=diagnostics, rois=rois if with_rois else None,
                                    fa_only=fa_only)
        want = _expected_volumes(shape, nt, plan.npc, n_bootstrap, parametric, diagnostics, with_rois, fa_only)
        assert set(vol) == set(want), opts
        for name, dt_shape in want.items():
            if dt_shape is None:
                assert isinstance(vol[name], dict), (name, opts)
            else:
                assert (vol[name].dtype, vol[name].shape) == dt_shape, (name, opts)


def test_host_buffers_keys_shapes_and_dtypes():
    plan = _plan()
    V = 100
    f64, i32 = torch.float64, torch.int32
    want = {"fsol": ((V, plan.npc), f64), "est_signal": ((V, 32), f64), "maps": ((V, 6), f64), "reg": ((V,), f64),
            "fa_deg": ((V,), f64), "fa_index": ((V,), i32), "km": ((V,), f64), "status": ((V,), i32),
            "fa_status": ((V,), i32), "fsol_sum": ((plan.npc,), f64)}
    boot = {"boot_stats": ((V, 6, 4), f64), "boot_n_valid": ((V,), i32)}
    param = {"param_params": ((V, 7), f64), "param_maps": ((V, 6), f64), "param_est_signal": ((V, 32), f64),
             "param_sse": ((V,), f64), "param_iters": ((V,), i32), "param_status": ((V,), i32)}
    for kw, extra in (({}, {}), (dict(n_bootstrap=8), boot), (dict(parametric=True), param),
                      (dict(n_bootstrap=8, parametric=True), {**boot, **param})):
        bufs = pipeline.host_buffers(plan, V, **kw)
        assert {k: (tuple(t.shape), t.dtype) for k, t in bufs.items()} == {**want, **extra}, kw
        assert all(t.is_pinned() for t in bufs.values())
    assert not any(t.is_pinned() for t in pipeline.host_buffers(plan, V, pinned=False).values())
