"""Plan-time instantiated kernels (vkfft_b200/csrc/jit.cpp): lengths outside the ahead-of-time lists get the hand-written
stockham.cuh templates compiled for them when their plan is created (NVRTC -> cubin), instead of the 3-5x slower
runtime-scheduled kernel.  CPU part: the kernel descriptions and the compile step (NVRTC needs no GPU).  GPU part: parity of
every kind of plan-time kernel against the oracle, tolerances of BASELINE.json's north_star (1e-6 / 1e-12 relative L2)."""
import ctypes
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "..", "oracle"))
import vkfft_oracle as orc

KIND_ROWS, KIND_TOUT, KIND_COLS = 0, 1, 2
OP_TW, OP_REAL_EVEN = 1, 16


def _lib():
    from vkfft_b200 import _lib
    L = _lib.load()
    L.b2_jit_selftest.restype = ctypes.c_long
    L.b2_jit_last_log.restype = ctypes.c_char_p
    return L


def _need_nvrtc(L):
    if not L.b2_jit_available():
        pytest.skip("libnvrtc not loadable here (or B200FFT_NO_JIT set): such lengths stay on the runtime-scheduled kernel")


@pytest.mark.parametrize("kind,prec,n,ops", [(KIND_ROWS, 0, 1100, 0), (KIND_ROWS, 0, 1430, OP_REAL_EVEN), (KIND_COLS, 0, 770, OP_TW),
                                             (KIND_COLS, 1, 154, 0), (KIND_TOUT, 0, 1100, 0), (KIND_ROWS, 1, 2002, 0),
                                             (KIND_ROWS, 0, 2 * 3 * 17, 0), (KIND_ROWS, 0, 4004, 0),
                                             (KIND_ROWS, 0, 1100, 32), (KIND_COLS, 1, 286, 32)])      # 32 = B2_OP_DCT23
def test_templates_compile_at_plan_time_without_a_gpu(kind, prec, n, ops):
    """the generated translation unit static_asserts the host-side copies of KCfg::SMEM_BYTES and RList::lut_size"""
    L = _lib()
    _need_nvrtc(L)
    size = L.b2_jit_selftest(kind, prec, n, ops)
    assert size > 10000, L.b2_jit_last_log().decode()[:2000]


@pytest.mark.parametrize("kind,prec,n,ops", [(KIND_ROWS, 0, 37, 0),          # prime: Bluestein
                                             (KIND_ROWS, 0, 17, 0),          # one radix: the staged short-line kernels
                                             (KIND_ROWS, 1, 34, 0),          # prime butterflies above 13 are FP32 only
                                             (KIND_COLS, 0, 4004, 0),        # strided tiles stop at 2048 points
                                             (KIND_ROWS, 0, 1100, 256),      # Bluestein launches are ahead-of-time only
                                             (KIND_ROWS, 0, 8200, 0),        # beyond one launch (8192 points)
                                             (KIND_ROWS, 1, 5000, 0)])       # FP64 stops at 4096
def test_keys_that_are_not_instantiated(kind, prec, n, ops):
    L = _lib()
    _need_nvrtc(L)
    assert L.b2_jit_selftest(kind, prec, n, ops) == 0


def test_plan_uses_a_plan_time_kernel_and_the_switch_turns_it_off(monkeypatch):
    """plan description without a GPU is not available (plans allocate tables on the device), so this checks the registry
    through the self test and the environment switch only"""
    L = _lib()
    _need_nvrtc(L)
    monkeypatch.setenv("B200FFT_NO_JIT", "1")
    assert L.b2_jit_available() == 0 and L.b2_jit_selftest(KIND_ROWS, 0, 1100, 0) == 0


def test_disk_cache_of_compiled_kernels(tmp_path):
    """B200FFT_JIT_CACHE=<dir>: the first process compiles and stores the cubin, the second one reads it back (same bytes, no
    compile) -- the saving the reference offers through saveApplicationToString / loadApplicationFromString"""
    import subprocess
    _need_nvrtc(_lib())
    code = ("import ctypes, sys, time; sys.path.insert(0, %r); from vkfft_b200 import _lib; L = _lib.load(); "
            "L.b2_jit_selftest.restype = ctypes.c_long; L.b2_jit_selftest(0, 0, 154, 0); t = time.time(); "
            "print(L.b2_jit_selftest(0, 0, 1430, 0), time.time() - t)") % os.path.join(os.path.dirname(__file__), "..")
    env = dict(os.environ, B200FFT_JIT_CACHE=str(tmp_path))
    first = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True).stdout.split()
    files = sorted(os.listdir(tmp_path))
    assert len(files) == 2 and all(f.endswith(".cubin") for f in files)
    sizes = {os.path.getsize(os.path.join(tmp_path, f)) for f in files}
    second = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True).stdout.split()
    assert int(first[0]) == int(second[0]) and int(first[0]) in sizes
    assert float(second[1]) < 0.25 * float(first[1]) + 0.05, (first, second)
    assert sorted(os.listdir(tmp_path)) == files


# ---------------------------------------------------------------- GPU ----------------------------------------------------------------
@pytest.fixture(scope="module")
def gpu():
    import torch
    assert torch.cuda.is_available(), "these tests need a GPU"
    import vkfft_b200  # noqa: F401  (fails loudly if libb200fft.so is missing)
    return torch


def _describe(vk, app):
    return " | ".join(vk.planInfo(app)["forward"]) if isinstance(vk.planInfo(app)["forward"], (list, tuple)) else str(vk.planInfo(app)["forward"])


@pytest.mark.gpu
@pytest.mark.parametrize("shape,batch,double", [((66,), 1000, False), ((154,), 77, False), ((1100,), 33, False), ((1430,), 9, False),
                                                ((2002,), 5, False), ((3003,), 3, False), ((4004,), 3, False), ((34,), 501, False),
                                                ((51,), 100, False), ((2 * 3 * 19 * 4,), 7, False), ((770,), 13, True), ((2002,), 3, True),
                                                ((1100, 154), 2, False), ((154, 66, 22), 2, False), ((286, 182), 2, True),
                                                ((1100 * 1430,), 1, False), ((2002 * 66,), 2, False),
                                                ((5000,), 3, False), ((6000,), 2, False), ((8190,), 2, False)])      # 4097...8192 points: one launch
@pytest.mark.parametrize("inverse", [-1, 1])
def test_c2c_lengths_without_ahead_of_time_kernels(gpu, shape, batch, double, inverse):
    """contiguous lines (ROWS), strided axes (COLS), Four-Step with such factors (COLS + phase, ROWS with transposed store)"""
    import torch
    import vkfft_b200 as vk
    L = _lib()
    _need_nvrtc(L)
    dt = np.complex128 if double else np.complex64
    x = orc.random_input((batch,) + tuple(reversed(shape)), dt, seed=sum(shape))
    t = torch.from_numpy(x).cuda()
    app = vk.VkFFTApplication()
    rc = vk.initializeVkFFT(app, vk.VkFFTConfiguration(FFTdim=len(shape), size=list(shape), numberBatches=batch, device=0, doublePrecision=int(double)))
    assert rc == 0, vk.getVkFFTErrorString(rc)
    try:
        desc = _describe(vk, app)
        assert "JIT_" in desc and "generic" not in desc, desc
        assert vk.VkFFTAppend(app, inverse, vk.VkFFTLaunchParams(buffer=t)) == 0
        torch.cuda.synchronize()
        got = t.cpu().numpy()
    finally:
        vk.deleteVkFFT(app)
    ref = orc.c2c(x, len(shape), inverse == 1)
    assert orc.error_metrics(got, ref)["l2_rel"] < (1e-12 if double else 1e-6)


@pytest.mark.gpu
@pytest.mark.parametrize("shape,batch,double", [((1100,), 5, False), ((2002, 6), 2, False), ((154, 22), 3, True), ((1430,), 4, True), ((14000,), 2, False)])
def test_r2c_c2r_lengths_without_ahead_of_time_kernels(gpu, shape, batch, double):
    """even-length real transforms: the Hermitian pass is fused into the plan-time kernel like into the ahead-of-time ones"""
    import torch
    import vkfft_b200 as vk
    L = _lib()
    _need_nvrtc(L)
    rdt = np.float64 if double else np.float32
    nx = shape[0]
    rs = (batch,) + tuple(reversed(shape[1:])) + (nx,)
    x = np.random.default_rng(sum(shape)).uniform(-1, 1, rs).astype(rdt)
    pad = np.zeros(rs[:-1] + (nx + 2,), rdt)
    pad[..., :nx] = x
    t = torch.from_numpy(pad).cuda()
    app = vk.VkFFTApplication()
    rc = vk.initializeVkFFT(app, vk.VkFFTConfiguration(FFTdim=len(shape), size=list(shape), numberBatches=batch, device=0, performR2C=1,
                                                       doublePrecision=int(double), normalize=1))
    assert rc == 0, vk.getVkFFTErrorString(rc)
    try:
        assert "JIT_" in _describe(vk, app)
        assert vk.VkFFTAppend(app, -1, vk.VkFFTLaunchParams(buffer=t)) == 0
        torch.cuda.synchronize()
        spec = t.cpu().numpy().view(np.complex128 if double else np.complex64)
        ref = np.fft.rfftn(x.astype(np.float64), axes=tuple(range(1, len(rs))))
        tol = 1e-12 if double else 1e-6
        assert orc.error_metrics(spec, ref)["l2_rel"] < tol
        assert vk.VkFFTAppend(app, 1, vk.VkFFTLaunchParams(buffer=t)) == 0
        torch.cuda.synchronize()
        back = t.cpu().numpy()[..., :nx]
        assert orc.error_metrics(back, x)["l2_rel"] < 2 * tol
    finally:
        vk.deleteVkFFT(app)


@pytest.mark.gpu
def test_switch_keeps_the_runtime_scheduled_kernel(gpu, monkeypatch):
    import torch
    import vkfft_b200 as vk
    monkeypatch.setenv("B200FFT_NO_JIT", "1")
    x = orc.random_input((5, 1100), np.complex64, seed=3)
    t = torch.from_numpy(x).cuda()
    app = vk.VkFFTApplication()
    assert vk.initializeVkFFT(app, vk.VkFFTConfiguration(FFTdim=1, size=[1100], numberBatches=5, device=0)) == 0
    try:
        assert "JIT_" not in _describe(vk, app)
        assert vk.VkFFTAppend(app, -1, vk.VkFFTLaunchParams(buffer=t)) == 0
        torch.cuda.synchronize()
        assert orc.error_metrics(t.cpu().numpy(), orc.c2c(x, 1))["l2_rel"] < 1e-6
    finally:
        vk.deleteVkFFT(app)


@pytest.mark.gpu
@pytest.mark.parametrize("shape,batch,double", [((1100,), 6, False), ((770, 154), 2, False), ((286, 22), 3, True), ((2310,), 2, False)])
@pytest.mark.parametrize("kind", [2, 3])
def test_dct_2_and_3_lengths_without_ahead_of_time_kernels(gpu, shape, batch, double, kind):
    """DCT-II / DCT-III fused into the plan-time kernels (two real lines per complex line; strided axes: pairs of columns)"""
    import torch
    import vkfft_b200 as vk
    L = _lib()
    _need_nvrtc(L)
    rdt = np.float64 if double else np.float32
    x = np.random.default_rng(sum(shape) + kind).uniform(-1, 1, (batch,) + tuple(reversed(shape))).astype(rdt)
    t = torch.from_numpy(x.copy()).cuda()
    app = vk.VkFFTApplication()
    rc = vk.initializeVkFFT(app, vk.VkFFTConfiguration(FFTdim=len(shape), size=list(shape), numberBatches=batch, device=0,
                                                       doublePrecision=int(double), performDCT=kind))
    assert rc == 0, vk.getVkFFTErrorString(rc)
    try:
        assert "JIT_" in _describe(vk, app)
        assert vk.VkFFTAppend(app, -1, vk.VkFFTLaunchParams(buffer=t)) == 0
        torch.cuda.synchronize()
        got = t.cpu().numpy()
    finally:
        vk.deleteVkFFT(app)
    ref = orc.dct(x, kind, len(shape))
    if double:
        assert orc.error_metrics(got, ref)["l2_rel"] < 1e-12
    else:      # 1e-6, or -- where the transform's conditioning puts both engines beyond it -- at least as close as the reference
        from gpu_util import assert_f32_parity
        assert_f32_parity(got, ref, x, shape, batch, -1, perform_dct=kind)
