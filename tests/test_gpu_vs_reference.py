"""GPU (-m gpu): same inputs through the engine and through the UNMODIFIED reference (CUDA backend, built into
oracle/_ref/libvkfft_ref.so by oracle/Makefile; what it computed on these inputs is stored in tests/golden/reference_gpu/cases.npz,
see gpu_util.reference).  North-star tolerance: 1e-6 rel FP32 / 1e-12 rel FP64.
The reference's default FP32 path evaluates twiddles with __sincosf (its own error vs FFTW is up to ~1.4e-6,
README.md:76-80), so the comparison is norm-wise, and also run against the reference with useLUT=1.
Distances to the reference's outputs are estimated from their stored sketches (gpu_util.sketch)."""
import numpy as np
import pytest

import vkfft_oracle as orc
from gpu_util import reference, sketch, sketch_l2_rel

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def torch():
    import torch
    assert torch.cuda.is_available()
    return torch


def _mine_c2c(size_xyz, batch, inverse, double):
    from gpu_util import run_c2c
    dt = np.complex128 if double else np.complex64
    x = orc.random_input((batch,) + tuple(reversed(size_xyz)), dt, seed=int(np.prod(size_xyz)) % 9973)
    return x, run_c2c(x, size_xyz, batch, inverse, double=double)


@pytest.mark.parametrize("n", [8, 128, 1024, 4096, 8192, 1 << 15, 1 << 18, 1 << 20, 1 << 23])
@pytest.mark.parametrize("inverse", [-1, 1])
def test_c2c_f32_matches_reference(torch, n, inverse):
    batch = max(1, (1 << 23) // n)
    x, mine = _mine_c2c((n,), batch, inverse, False)
    sk_m = sketch(mine)
    assert sketch_l2_rel(sk_m, reference(x, (n,), batch, inverse, use_lut=1)["sketch"]) < 1e-6
    # reference default (on-chip sincos) carries its own ~1e-6 error for large N; both must sit within 1e-6 of
    # the exact result's neighbourhood: |mine - theirs| <= |mine - exact| + |theirs - exact|
    exact = orc.c2c(x, 1, inverse == 1)
    theirs = reference(x, (n,), batch, inverse, use_lut=0, exact=exact)
    e_m = orc.error_metrics(mine, exact)["l2_rel"]
    e_t = theirs["l2_exact"]
    assert e_m < 1e-6 and e_m <= e_t * 1.05 + 1e-8
    sk_t, sk_e = theirs["sketch"], sketch(exact)
    assert sketch_l2_rel(sk_m, sk_t) < sketch_l2_rel(sk_m, sk_e) + sketch_l2_rel(sk_t, sk_e) + 1e-9


@pytest.mark.parametrize("size_xyz", [(4096,), (1 << 16,), (256, 256, 256)])
def test_c2c_f64_matches_reference(torch, size_xyz):
    x, mine = _mine_c2c(size_xyz, 1, -1, True)
    assert sketch_l2_rel(sketch(mine), reference(x, size_xyz, 1, -1, double=True, use_lut=0)["sketch"]) < 1e-12


def _mine_inplace(torch, arr, size_xyz, batch, inverse, double=False, **kw):
    import vkfft_b200 as vk
    t = torch.from_numpy(np.ascontiguousarray(arr)).cuda()
    app = vk.VkFFTApplication()
    cfg = vk.VkFFTConfiguration(FFTdim=len(size_xyz), size=list(size_xyz), numberBatches=batch, device=0,
                                doublePrecision=int(double), **kw)
    rc = vk.initializeVkFFT(app, cfg)
    assert rc == 0, vk.getVkFFTErrorString(rc)
    try:
        assert vk.VkFFTAppend(app, inverse, vk.VkFFTLaunchParams(buffer=t)) == 0
        torch.cuda.synchronize()
        return t.cpu().numpy()
    finally:
        vk.deleteVkFFT(app)


@pytest.mark.parametrize("size_xyz,batch", [((1000,), 8), ((2187,), 3), ((30030,), 2), ((17,), 64), ((509,), 8), ((105, 30), 2)])
@pytest.mark.parametrize("inverse", [-1, 1])
def test_non_pow2_matches_reference(torch, size_xyz, batch, inverse):
    x = orc.random_input((batch,) + tuple(reversed(size_xyz)), np.complex64, seed=sum(size_xyz))
    mine = _mine_inplace(torch, x, size_xyz, batch, inverse)
    assert sketch_l2_rel(sketch(mine), reference(x, size_xyz, batch, inverse)["sketch"]) < 1e-6


@pytest.mark.parametrize("size_xyz,batch", [((64,), 8), ((4096,), 4), ((4096, 4096), 1), ((30, 4), 3)])
def test_r2c_c2r_matches_reference(torch, size_xyz, batch):
    nx, H = size_xyz[0], size_xyz[0] // 2 + 1
    x = orc.random_input((batch,) + tuple(reversed(size_xyz)), np.float32, seed=sum(size_xyz))
    buf = np.zeros(x.shape[:-1] + (2 * H,), np.float32)
    buf[..., :nx] = x
    mine = _mine_inplace(torch, buf, size_xyz, batch, -1, performR2C=1)
    theirs = reference(buf, size_xyz, batch, -1, perform_r2c=1)["sketch"]
    assert sketch_l2_rel(sketch(mine), theirs) < 1e-6
    # C2R of the same Hermitian half-spectrum through both engines: the exact one, rounded to FP32
    spec = orc.r2c(x, len(size_xyz)).astype(np.complex64).view(np.float32)
    mine2 = _mine_inplace(torch, spec, size_xyz, batch, 1, performR2C=1)
    theirs2 = reference(spec, size_xyz, batch, 1, crop=nx, perform_r2c=1)["sketch"]
    assert sketch_l2_rel(sketch(mine2[..., :nx]), theirs2) < 1e-6


@pytest.mark.parametrize("kind", [1, 2, 3, 4])
@pytest.mark.parametrize("size_xyz,batch", [((64,), 6), ((100,), 4), ((32, 16), 3), ((2048, 256), 1)])
@pytest.mark.parametrize("inverse", [-1, 1])
def test_dct_matches_reference(torch, kind, size_xyz, batch, inverse):
    x = orc.random_input((batch,) + tuple(reversed(size_xyz)), np.float32, seed=kind + sum(size_xyz))
    mine = _mine_inplace(torch, x, size_xyz, batch, inverse, performDCT=kind)
    exact = orc.dct(x, kind, len(size_xyz), inverse=(inverse == 1))
    theirs = reference(x, size_xyz, batch, inverse, exact=exact, perform_dct=kind)
    # north-star 1e-6 between the two engines; where the transform's conditioning puts the reference itself further than
    # that from the exact result, this engine must be at least as close to it as the reference is
    sk_m, sk_t = sketch(mine), theirs["sketch"]
    d = sketch_l2_rel(sk_m, sk_t)
    if d >= 1e-6:
        sk_e = sketch(exact)
        e_m = orc.error_metrics(mine, exact)["l2_rel"]
        e_t = theirs["l2_exact"]
        assert e_m <= 1.05 * e_t + 1e-8 and d < sketch_l2_rel(sk_m, sk_e) + sketch_l2_rel(sk_t, sk_e) + 1e-9, (d, e_m, e_t)
