"""batched.noise_sigma / batched.tv_denoise (met2_noise_sigma, met2_tv_chambolle) on the device, bitwise equal to the
NumPy restatement of tests/tv_oracle.py on the 96 x 96 x 60 x 32 phantom, masked like the orchestrator does."""
import numpy as np
import pytest

import tv_oracle as T


@pytest.fixture(scope="module")
def phantom():
    from multicomponent_t2_toolbox_b200.phantom import make_phantom
    ph = make_phantom((96, 96, 60), seed=2, fa_mode="b1", mask_mode="ellipsoid", backend="gpu")
    data = ph["data"] * ph["mask"][..., None]          # motor_recon_met2: data * mask, negatives clipped
    data[data < 0.0] = 0.0
    return np.ascontiguousarray(data)


@pytest.mark.gpu
def test_noise_sigma_bitwise_for_every_echo(phantom):
    from multicomponent_t2_toolbox_b200 import batched
    s = batched.noise_sigma(phantom).cpu().numpy()
    ref = np.array([T.estimate_sigma(phantom[..., t]) for t in range(phantom.shape[3])])
    assert np.isfinite(ref).all() and np.array_equal(s, ref)


@pytest.mark.gpu
def test_tv_full_size_first_and_last_echo(phantom):
    from multicomponent_t2_toolbox_b200 import batched
    sub = np.ascontiguousarray(phantom[..., [0, 31]])
    out, iters = batched.tv_denoise(sub)
    out, iters = out.cpu().numpy(), iters.cpu().numpy()
    for k in range(2):
        vol = sub[..., k]
        ref, it = T.denoise_tv_chambolle(vol, 2.0 * T.estimate_sigma(vol))
        assert iters[k] == it and np.array_equal(out[..., k], ref)


@pytest.mark.gpu
def test_tv_every_echo_on_a_crop(phantom):
    from multicomponent_t2_toolbox_b200 import batched
    crop = np.ascontiguousarray(phantom[24:72, 24:72, 15:45])
    ref, sigma, iters = T.tv_denoise(crop)
    out, it = batched.tv_denoise(crop)
    assert np.array_equal(it.cpu().numpy(), iters)
    assert np.array_equal(out.cpu().numpy(), ref)


@pytest.mark.gpu
def test_tv_single_slice(phantom):
    from multicomponent_t2_toolbox_b200 import batched
    sl = np.ascontiguousarray(phantom[:, :, 30:31])
    ref, sigma, iters = T.tv_denoise(sl)
    out, it = batched.tv_denoise(sl)
    assert np.array_equal(batched.noise_sigma(sl).cpu().numpy(), sigma)
    assert np.array_equal(it.cpu().numpy(), iters)
    assert np.array_equal(out.cpu().numpy(), ref)


@pytest.mark.gpu
def test_tv_repeatable_and_explicit_weights(phantom):
    import torch
    from multicomponent_t2_toolbox_b200 import batched
    data = torch.as_tensor(phantom).cuda()
    a, ia = batched.tv_denoise(data)
    b, ib = batched.tv_denoise(data)
    assert torch.equal(a, b) and torch.equal(ia, ib)
    w = 2.0 * batched.noise_sigma(data)
    c, ic = batched.tv_denoise(data, weight=w.cpu().numpy().tolist())
    assert torch.equal(a, c) and torch.equal(ia, ic)
