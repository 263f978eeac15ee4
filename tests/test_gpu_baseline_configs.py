"""GPU (-m gpu): BASELINE.json configs 3, 4 and 5 AT THEIR FULL SIZES against the oracle, and performZeropadding.

  config 3   3-D C2C FP64 512^3 (256^3 is in test_gpu_parity / test_gpu_vs_reference): the whole result against pocketfft
  config 4   2-D DCT-II 8192 x 8192 FP32: the whole result against the oracle, and the DCT-III round trip
  config 5   1-D C2C FP32 N = 2^26 (the three-launch Four-Step at the size the config names): every sequence of a batch of 2
             against the oracle, Parseval, round trip
  zero padding  the shapes of the reference's samples 4 and 51 (open systems: the upper half of every axis is padding)
Tolerances: 1e-6 relative l2 FP32 (composed real transforms: the stated inequality against the reference, gpu_util.py),
1e-12 FP64."""
import numpy as np
import pytest

import vkfft_oracle as orc

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def gpu():
    import torch
    assert torch.cuda.is_available(), "these tests need a GPU"
    return torch


def _run(torch, arr, inverse, **cfgkw):
    import vkfft_b200 as vk
    t = torch.from_numpy(np.ascontiguousarray(arr)).cuda()
    app = vk.VkFFTApplication()
    rc = vk.initializeVkFFT(app, vk.VkFFTConfiguration(device=0, **cfgkw))
    assert rc == 0, vk.getVkFFTErrorString(rc)
    try:
        assert vk.VkFFTAppend(app, inverse, vk.VkFFTLaunchParams(buffer=t)) == 0
        torch.cuda.synchronize()
        return t.cpu().numpy()
    finally:
        vk.deleteVkFFT(app)


@pytest.mark.parametrize("inverse", [-1, 1])
def test_config3_c2c_fp64_512_cubed(gpu, inverse):
    n = 512
    x = orc.random_input((1, n, n, n), np.complex128, seed=512 + inverse)
    y = _run(gpu, x, inverse, FFTdim=3, size=[n, n, n], numberBatches=1, doublePrecision=1)
    assert orc.error_metrics(y, orc.c2c(x, 3, inverse == 1))["l2_rel"] < 1e-12


def test_config4_dct2_fp32_8192_squared(gpu):
    from gpu_util import assert_f32_parity
    n = 8192
    x = orc.random_input((1, n, n), np.float32, seed=8192)
    y = _run(gpu, x, -1, FFTdim=2, size=[n, n], numberBatches=1, performDCT=2)
    exact = orc.dct(x, 2, 2)
    assert_f32_parity(y, exact, x, (n, n), 1, -1, perform_dct=2)
    # DCT-III of the result returns (2n)^2 x  (API guide: unnormalised pair)
    z = _run(gpu, y, 1, FFTdim=2, size=[n, n], numberBatches=1, performDCT=2)
    assert orc.error_metrics(z, x.astype(np.float64) * (2.0 * n) ** 2)["l2_rel"] < 2e-6


def test_config5_c2c_fp32_2_pow_26(gpu):
    torch = gpu
    import vkfft_b200 as vk
    n, batch = 1 << 26, 2
    x = orc.random_input((batch, n), np.complex64, seed=26)
    t = torch.from_numpy(x).cuda()
    app = vk.VkFFTApplication()
    assert vk.initializeVkFFT(app, vk.VkFFTConfiguration(FFTdim=1, size=[n], numberBatches=batch, device=0)) == 0
    try:
        assert vk.planInfo(app)["num_passes_forward"] >= 2
        assert vk.VkFFTAppend(app, -1, vk.VkFFTLaunchParams(buffer=t)) == 0
        torch.cuda.synchronize()
        y = t.cpu().numpy()
        assert orc.error_metrics(y, orc.c2c(x, 1))["l2_rel"] < 1e-6
        e_in = float((np.abs(x.astype(np.complex128)) ** 2).sum())
        e_out = float((np.abs(y.astype(np.complex128)) ** 2).sum())
        assert abs(e_out / (n * e_in) - 1) < 1e-5                      # Parseval
        assert vk.VkFFTAppend(app, 1, vk.VkFFTLaunchParams(buffer=t)) == 0
        torch.cuda.synchronize()
        z = t.cpu().numpy()
        assert orc.error_metrics(z, x.astype(np.complex128) * n)["l2_rel"] < 2e-6
    finally:
        vk.deleteVkFFT(app)


# ---- performZeropadding (API guide :1786-1807; samples 4 and 51) ---------------------------------------------------------
def test_zero_padding_c2c_3d_open_system_sample_4_shape(gpu):
    """sample_4_benchmark_VkFFT_single_3d_zeropadding.cpp: the upper half of every axis is padding; whatever the buffer holds
    there, the transform must act on zeros"""
    rng = np.random.default_rng(4)
    n = 64
    x = (rng.uniform(-1, 1, (2, n, n, n)) + 1j * rng.uniform(-1, 1, (2, n, n, n))).astype(np.complex64)
    clean = x.copy()
    clean[..., n // 2:] = 0; clean[:, :, n // 2:, :] = 0; clean[:, n // 2:, :, :] = 0
    y = _run(gpu, x, -1, FFTdim=3, size=[n, n, n], numberBatches=2, performZeropadding=[1, 1, 1],
             fft_zeropad_left=[n // 2] * 3, fft_zeropad_right=[n] * 3)
    assert orc.error_metrics(y, orc.c2c(clean, 3))["l2_rel"] < 1e-6


def test_zero_padding_r2c_2d(gpu):
    rng = np.random.default_rng(51)
    nx, ny, b = 256, 96, 3
    x = rng.uniform(-1, 1, (b, ny, nx)).astype(np.float32)
    clean = x.copy()
    clean[..., nx // 2:] = 0; clean[:, ny // 2:, :] = 0
    buf = np.full((b, ny, nx + 2), 7.0, np.float32)
    buf[..., :nx] = x
    y = _run(gpu, buf, -1, FFTdim=2, size=[nx, ny], numberBatches=b, performR2C=1, performZeropadding=[1, 1],
             fft_zeropad_left=[nx // 2, ny // 2], fft_zeropad_right=[nx, ny])
    assert orc.error_metrics(y.view(np.complex64), orc.r2c(clean, 2))["l2_rel"] < 1e-6


def test_zero_padding_long_axis_and_frequency_padding(gpu):
    rng = np.random.default_rng(7)
    n, b = 1 << 16, 3                          # a Four-Step axis (fused launch) behind the clearing pass
    x = (rng.uniform(-1, 1, (b, n)) + 1j * rng.uniform(-1, 1, (b, n))).astype(np.complex64)
    clean = x.copy()
    clean[:, n // 4: n // 2] = 0
    y = _run(gpu, x, -1, FFTdim=1, size=[n], numberBatches=b, performZeropadding=[1], fft_zeropad_left=[n // 4],
             fft_zeropad_right=[n // 2])
    assert orc.error_metrics(y, orc.c2c(clean, 1))["l2_rel"] < 1e-6
    # frequencyZeroPadding: the forward transform is untouched, the inverse reads zeros in the flagged range
    y = _run(gpu, x, -1, FFTdim=1, size=[n], numberBatches=b, performZeropadding=[1], fft_zeropad_left=[n // 4],
             fft_zeropad_right=[n // 2], frequencyZeroPadding=1)
    assert orc.error_metrics(y, orc.c2c(x, 1))["l2_rel"] < 1e-6
    z = _run(gpu, x, 1, FFTdim=1, size=[n], numberBatches=b, performZeropadding=[1], fft_zeropad_left=[n // 4],
             fft_zeropad_right=[n // 2], frequencyZeroPadding=1)
    assert orc.error_metrics(z, orc.c2c(clean, 1, True))["l2_rel"] < 1e-6
