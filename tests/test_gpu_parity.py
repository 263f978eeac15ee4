"""GPU (-m gpu): parity of the CUDA path, called through the C ABI, against the double-precision oracle on
seeded inputs, plus size-independent properties at BASELINE.json's full sizes.
Tolerances (BASELINE.json north_star): 1e-6 relative FP32, 1e-12 relative FP64 (norm-wise L2)."""
import numpy as np
import pytest

import vkfft_oracle as orc

pytestmark = pytest.mark.gpu

TOL32, TOL64 = 1e-6, 1e-12


@pytest.fixture(scope="module")
def gpu():
    import torch
    assert torch.cuda.is_available(), "these tests need a GPU"
    import vkfft_b200  # noqa: F401  (fails loudly if libb200fft.so is missing)
    from vkfft_b200 import _lib
    assert _lib.load().b200fft_kernel_count() > 0
    return torch


POW2 = [2 ** k for k in range(1, 23)]


@pytest.mark.parametrize("n", POW2)
@pytest.mark.parametrize("inverse", [-1, 1])
def test_c2c_1d_f32_vs_oracle(gpu, n, inverse):
    from gpu_util import run_c2c
    batch = max(1, min(37, (1 << 22) // n))          # odd batch: exercises ragged line groups
    x = orc.random_input((batch, n), np.complex64, seed=n)
    got = run_c2c(x, (n,), batch, inverse)
    ref = orc.c2c(x, 1, inverse == 1)
    assert orc.error_metrics(got, ref)["l2_rel"] < TOL32


@pytest.mark.parametrize("n", [2 ** k for k in range(1, 21)])
@pytest.mark.parametrize("inverse", [-1, 1])
def test_c2c_1d_f64_vs_oracle(gpu, n, inverse):
    from gpu_util import run_c2c
    batch = max(1, min(19, (1 << 20) // n))
    x = orc.random_input((batch, n), np.complex128, seed=n + 7)
    got = run_c2c(x, (n,), batch, inverse, double=True)
    ref = orc.c2c(x, 1, inverse == 1)
    assert orc.error_metrics(got, ref)["l2_rel"] < TOL64


@pytest.mark.parametrize("shape_xyz,double", [((64, 32), False), ((256, 256), False), ((128, 64, 32), False),
                                              ((64, 64, 64), True), ((256, 256, 256), True), ((16, 8, 4, 2), False),
                                              ((4096, 64), False), ((32, 2048), False)])
@pytest.mark.parametrize("inverse", [-1, 1])
def test_c2c_nd_vs_oracle(gpu, shape_xyz, double, inverse):
    from gpu_util import run_c2c
    batch = 2 if np.prod(shape_xyz) < (1 << 22) else 1
    dt = np.complex128 if double else np.complex64
    x = orc.random_input((batch,) + tuple(reversed(shape_xyz)), dt, seed=sum(shape_xyz))
    got = run_c2c(x, shape_xyz, batch, inverse, double=double)
    ref = orc.c2c(x, len(shape_xyz), inverse == 1)
    assert orc.error_metrics(got, ref)["l2_rel"] < (TOL64 if double else TOL32)


def test_normalize_and_round_trip(gpu):
    from gpu_util import run_c2c
    n, batch = 4096, 8
    x = orc.random_input((batch, n), np.complex64, 3)
    y = run_c2c(x, (n,), batch, -1)
    z = run_c2c(y, (n,), batch, 1, normalize=1)
    assert orc.error_metrics(z, x)["l2_rel"] < TOL32
    z2 = run_c2c(y, (n,), batch, 1)
    assert orc.error_metrics(z2, n * x.astype(np.complex128))["l2_rel"] < TOL32


def test_known_answer_vectors(gpu):
    from gpu_util import run_c2c
    for n in (8, 4096, 1 << 16):
        e = np.zeros((2, n), np.complex64)
        e[0, 0] = 1
        e[1, 5] = 1
        y = run_c2c(e, (n,), 2, -1)
        k = np.arange(n)
        assert np.allclose(y[0], 1, atol=1e-6)
        assert np.allclose(y[1], np.exp(-2j * np.pi * 5 * k / n), atol=2e-6)


@pytest.mark.parametrize("n", [1 << 12, 1 << 17, 1 << 20, 1 << 22])
def test_full_size_properties_2gib(gpu, n):
    """BASELINE config 2 at full size (2 GiB buffer): too big for the CPU oracle, so check properties that pin
    the transform: inverse(forward(x)) == N x, Parseval, and exact agreement with the oracle on a few sequences."""
    torch = gpu
    import vkfft_b200 as vk
    total = 1 << 28
    batch = total // n
    g = torch.Generator(device="cuda").manual_seed(n)
    x = torch.empty((batch, n, 2), dtype=torch.float32, device="cuda").uniform_(-1, 1, generator=g)
    x0 = x.clone()
    app = vk.VkFFTApplication()
    assert vk.initializeVkFFT(app, vk.VkFFTConfiguration(FFTdim=1, size=[n], numberBatches=batch, device=0)) == 0
    try:
        assert vk.VkFFTAppend(app, -1, vk.VkFFTLaunchParams(buffer=x)) == 0
        torch.cuda.synchronize()
        # spot-check a few sequences against the CPU oracle
        for b in (0, batch // 2, batch - 1):
            xin = torch.view_as_complex(x0[b]).cpu().numpy()[None]
            got = torch.view_as_complex(x[b]).cpu().numpy()[None]
            assert orc.error_metrics(got, orc.c2c(xin, 1))["l2_rel"] < TOL32
        # Parseval: sum |X|^2 = N sum |x|^2
        e_in = (x0.double() ** 2).sum().item()
        e_out = (x.double() ** 2).sum().item()
        assert abs(e_out / (n * e_in) - 1) < 1e-5
        assert vk.VkFFTAppend(app, 1, vk.VkFFTLaunchParams(buffer=x)) == 0
        torch.cuda.synchronize()
        x.mul_(1.0 / n)
        err = (x - x0).double().norm().item() / x0.double().norm().item()
        assert err < 2e-6
    finally:
        vk.deleteVkFFT(app)


def test_api_errors_on_gpu(gpu):
    import vkfft_b200 as vk
    app = vk.VkFFTApplication()
    assert vk.initializeVkFFT(app, vk.VkFFTConfiguration(FFTdim=0, size=[8], device=0)) == vk.VKFFT_ERROR_EMPTY_FFTdim
    assert vk.initializeVkFFT(app, vk.VkFFTConfiguration(FFTdim=1, size=[0], device=0)) == vk.VKFFT_ERROR_EMPTY_size
    assert vk.initializeVkFFT(app, vk.VkFFTConfiguration(FFTdim=1, size=[8], device=99)) == vk.VKFFT_ERROR_INVALID_DEVICE
    assert vk.initializeVkFFT(app, vk.VkFFTConfiguration(FFTdim=1, size=[8], device=0, makeForwardPlanOnly=1)) == 0
    t = gpu.zeros(8, dtype=gpu.complex64, device="cuda")
    assert vk.VkFFTAppend(app, 1, vk.VkFFTLaunchParams(buffer=t)) == vk.VKFFT_ERROR_ONLY_FORWARD_FFT_INITIALIZED
    assert vk.VkFFTAppend(app, -1, vk.VkFFTLaunchParams()) == vk.VKFFT_ERROR_EMPTY_buffer
    assert vk.initializeVkFFT(app, vk.VkFFTConfiguration(FFTdim=1, size=[8], device=0)) == vk.VKFFT_ERROR_NONZERO_APP_INITIALIZATION
    vk.deleteVkFFT(app)
    assert vk.VkFFTAppend(app, -1, vk.VkFFTLaunchParams(buffer=t)) == vk.VKFFT_ERROR_PLAN_NOT_INITIALIZED


# ---- the runtime-scheduled kernel and its fused operators ------------------------------------------------------------
@pytest.mark.parametrize("shape,batch,double", [((1000,), 33, False), ((2187,), 5, False), ((77,), 50, True),
                                                ((30030,), 3, False), ((105, 30), 4, False), ((7, 11, 13), 3, True),
                                                ((17,), 100, False), ((509,), 9, False), ((1019,), 3, True),
                                                ((23, 8), 5, False), ((4093,), 2, False), ((3 ** 8,), 2, False),
                                                ((5 ** 5,), 3, True), ((7 ** 4,), 3, False), ((11 ** 3,), 3, False),
                                                ((13 ** 3,), 3, False), ((2 * 3 * 5 * 7 * 11 * 13 * 4,), 1, False),
                                                ((127,), 40, False), ((1088,), 9, False), ((2032,), 5, True), ((94,), 33, False),
                                                ((12167,), 2, False), ((131,), 30, False), ((8, 139), 3, True)])
@pytest.mark.parametrize("inverse", [-1, 1])
def test_c2c_non_pow2_and_bluestein(gpu, shape, batch, double, inverse):
    from gpu_util import run_c2c
    dt = np.complex128 if double else np.complex64
    x = orc.random_input((batch,) + tuple(reversed(shape)), dt, seed=sum(shape))
    got = run_c2c(x, shape, batch, inverse, double=double)
    ref = orc.c2c(x, len(shape), inverse == 1)
    assert orc.error_metrics(got, ref)["l2_rel"] < (TOL64 if double else TOL32)


def _smooth13(n):
    for p in [2, 3, 5, 7, 11, 13] + [q for q in range(17, 128, 2) if all(q % r for r in range(3, 12, 2))]:
        while n % p == 0:
            n //= p
    return n == 1


def _run_plan(torch, arr, cfg, inverse):
    import vkfft_b200 as vk
    t = torch.from_numpy(np.ascontiguousarray(arr)).cuda()
    app = vk.VkFFTApplication()
    rc = vk.initializeVkFFT(app, cfg)
    assert rc == 0, vk.getVkFFTErrorString(rc)
    try:
        assert vk.VkFFTAppend(app, inverse, vk.VkFFTLaunchParams(buffer=t)) == 0
        torch.cuda.synchronize()
        return t.cpu().numpy()
    finally:
        vk.deleteVkFFT(app)


@pytest.mark.parametrize("shape,batch,double", [((64,), 7, False), ((4096,), 5, False), ((4096, 4096), 1, False),
                                                ((30,), 3, True), ((15,), 3, False), ((128, 8, 4), 2, True),
                                                ((1000, 6), 2, False), ((8192,), 3, False), ((131,), 3, False), ((4391,), 2, False),
                                                ((263, 5), 2, True)])
def test_r2c_c2r(gpu, shape, batch, double):
    import vkfft_b200 as vk
    rdt, cdt = (np.float64, np.complex128) if double else (np.float32, np.complex64)
    tol = TOL64 if double else TOL32
    nx, H = shape[0], shape[0] // 2 + 1
    x = orc.random_input((batch,) + tuple(reversed(shape)), rdt, seed=sum(shape))
    buf = np.zeros(x.shape[:-1] + (2 * H,), rdt)
    buf[..., :nx] = x
    cfg = vk.VkFFTConfiguration(FFTdim=len(shape), size=list(shape), numberBatches=batch, device=0, performR2C=1,
                                doublePrecision=int(double))
    y = _run_plan(gpu, buf, cfg, -1)
    assert orc.error_metrics(y.view(cdt), orc.r2c(x, len(shape)))["l2_rel"] < tol
    z = _run_plan(gpu, y, cfg, 1)
    assert orc.error_metrics(z[..., :nx], x.astype(np.float64) * np.prod(shape))["l2_rel"] < tol


@pytest.mark.parametrize("kind", [1, 2, 3, 4])
@pytest.mark.parametrize("shape,batch,double", [((64,), 5, False), ((33,), 4, True), ((32, 16), 3, False), ((100,), 3, True),
                                                ((8, 6, 4), 2, False), ((4096,), 3, False), ((1024, 512), 1, False),
                                                ((64, 8192), 1, False), ((2048, 4096), 1, False), ((63, 256), 2, True)])
@pytest.mark.parametrize("inverse", [-1, 1])
def test_dct(gpu, kind, shape, batch, double, inverse):
    import vkfft_b200 as vk
    from gpu_util import assert_f32_parity
    rdt = np.float64 if double else np.float32
    x = orc.random_input((batch,) + tuple(reversed(shape)), rdt, seed=kind + sum(shape))
    cfg = vk.VkFFTConfiguration(FFTdim=len(shape), size=list(shape), numberBatches=batch, device=0, performDCT=kind,
                                doublePrecision=int(double))
    y = _run_plan(gpu, x, cfg, inverse)
    ref = orc.dct(x, kind, len(shape), inverse=(inverse == 1))
    if double:
        assert orc.error_metrics(y, ref)["l2_rel"] < TOL64
    else:
        assert_f32_parity(y, ref, x, shape, batch, inverse, perform_dct=kind)


def test_out_of_place_formatted_buffers(gpu):
    """isInputFormatted / isOutputFormatted plumbing (API guide :365-376) for C2C and R2C"""
    import vkfft_b200 as vk
    torch = gpu
    n, batch = 1024, 6
    x = orc.random_input((batch, n), np.complex64, 11)
    tin = torch.from_numpy(x).cuda()
    tbuf = torch.zeros_like(tin)
    tout = torch.zeros_like(tin)
    app = vk.VkFFTApplication()
    cfg = vk.VkFFTConfiguration(FFTdim=1, size=[n], numberBatches=batch, device=0, isInputFormatted=1, isOutputFormatted=1)
    assert vk.initializeVkFFT(app, cfg) == 0
    assert vk.VkFFTAppend(app, -1, vk.VkFFTLaunchParams(buffer=tbuf, inputBuffer=tin, outputBuffer=tout)) == 0
    torch.cuda.synchronize()
    assert orc.error_metrics(tout.cpu().numpy(), orc.c2c(x, 1))["l2_rel"] < TOL32
    assert np.array_equal(tin.cpu().numpy(), x)          # input untouched
    vk.deleteVkFFT(app)
    # R2C from an unpadded real input buffer
    xr = orc.random_input((batch, 16, 64), np.float32, 12)
    tr = torch.from_numpy(xr).cuda()
    tc = torch.zeros((batch, 16, 33), dtype=torch.complex64, device="cuda")
    app = vk.VkFFTApplication()
    cfg = vk.VkFFTConfiguration(FFTdim=2, size=[64, 16], numberBatches=batch, device=0, performR2C=1, isInputFormatted=1,
                                inverseReturnToInputBuffer=1)
    assert vk.initializeVkFFT(app, cfg) == 0
    assert vk.VkFFTAppend(app, -1, vk.VkFFTLaunchParams(buffer=tc, inputBuffer=tr)) == 0
    torch.cuda.synchronize()
    assert orc.error_metrics(tc.cpu().numpy(), orc.r2c(xr, 2))["l2_rel"] < TOL32
    tr.zero_()
    assert vk.VkFFTAppend(app, 1, vk.VkFFTLaunchParams(buffer=tc, inputBuffer=tr)) == 0
    torch.cuda.synchronize()
    assert orc.error_metrics(tr.cpu().numpy(), xr.astype(np.float64) * 64 * 16)["l2_rel"] < TOL32
    vk.deleteVkFFT(app)


@pytest.mark.parametrize("kind", [1, 2, 3, 4])
@pytest.mark.parametrize("shape,batch,double", [((64,), 5, False), ((32, 16), 3, False), ((100,), 3, True), ((4096,), 2, False),
                                                ((33,), 4, True), ((45, 21), 2, False)])
@pytest.mark.parametrize("inverse", [-1, 1])
def test_dst(gpu, kind, shape, batch, double, inverse):
    import vkfft_b200 as vk
    from gpu_util import assert_f32_parity
    rdt = np.float64 if double else np.float32
    x = orc.random_input((batch,) + tuple(reversed(shape)), rdt, seed=kind + sum(shape))
    cfg = vk.VkFFTConfiguration(FFTdim=len(shape), size=list(shape), numberBatches=batch, device=0, performDST=kind,
                                doublePrecision=int(double))
    y = _run_plan(gpu, x, cfg, inverse)
    ref = orc.dst(x, kind, len(shape), inverse=(inverse == 1))
    if double:
        assert orc.error_metrics(y, ref)["l2_rel"] < TOL64
    else:
        assert_f32_parity(y, ref, x, shape, batch, inverse, perform_dst=kind)


@pytest.mark.parametrize("shape,batch,double", [((1 << 20,), 3, False), ((2 * 4391,), 4, False), ((1 << 17, 4), 1, True)])
def test_long_r2c_c2r(gpu, shape, batch, double):
    import vkfft_b200 as vk
    rdt, cdt = (np.float64, np.complex128) if double else (np.float32, np.complex64)
    tol = TOL64 if double else TOL32
    nx, H = shape[0], shape[0] // 2 + 1
    x = orc.random_input((batch,) + tuple(reversed(shape)), rdt, seed=sum(shape))
    buf = np.zeros(x.shape[:-1] + (2 * H,), rdt)
    buf[..., :nx] = x
    cfg = vk.VkFFTConfiguration(FFTdim=len(shape), size=list(shape), numberBatches=batch, device=0, performR2C=1,
                                doublePrecision=int(double))
    y = _run_plan(gpu, buf, cfg, -1)
    assert orc.error_metrics(y.view(cdt), orc.r2c(x, len(shape)))["l2_rel"] < tol
    z = _run_plan(gpu, y, cfg, 1)
    assert orc.error_metrics(z[..., :nx], x.astype(np.float64) * np.prod(shape))["l2_rel"] < tol


@pytest.mark.parametrize("shape,batch,double", [((4391,), 6, False), ((20011,), 2, False), ((5003,), 2, True), ((16, 8192), 2, False),
                                                ((100003,), 1, False)])
@pytest.mark.parametrize("inverse", [-1, 1])
def test_long_bluestein_and_strided_four_step(gpu, shape, batch, double, inverse):
    from gpu_util import run_c2c
    dt = np.complex128 if double else np.complex64
    x = orc.random_input((batch,) + tuple(reversed(shape)), dt, seed=sum(shape))
    got = run_c2c(x, shape, batch, inverse, double=double)
    assert orc.error_metrics(got, orc.c2c(x, len(shape), inverse == 1))["l2_rel"] < (TOL64 if double else TOL32)


def test_pipelined_kernels_fall_back_on_unaligned_buffers(gpu):
    """the TMA-fed kernels (N=16384 single pass, transposed 2048) need 16-byte aligned sources; with an 8-byte
    bufferOffset the engine must switch to the plain kernels (and their own twiddle tables)"""
    import vkfft_b200 as vk
    torch = gpu
    for n in (16384, 1 << 16, 1 << 22):
        batch = max(1, (1 << 22) // n) if n < (1 << 22) else 1
        x = orc.random_input((batch, n), np.complex64, seed=n + 5)
        raw = torch.zeros(batch * n + 1, dtype=torch.complex64, device="cuda")
        raw[1:] = torch.from_numpy(x.reshape(-1)).cuda()
        app = vk.VkFFTApplication()
        assert vk.initializeVkFFT(app, vk.VkFFTConfiguration(FFTdim=1, size=[n], numberBatches=batch, device=0,
                                                             specifyOffsetsAtLaunch=1)) == 0
        assert vk.VkFFTAppend(app, -1, vk.VkFFTLaunchParams(buffer=raw, bufferOffset=8)) == 0
        torch.cuda.synchronize()
        got = raw[1:].cpu().numpy().reshape(batch, n)
        vk.deleteVkFFT(app)
        assert orc.error_metrics(got, orc.c2c(x, 1))["l2_rel"] < TOL32
