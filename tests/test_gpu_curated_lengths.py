"""GPU (-m gpu): every line of csrc/kernel_list_nonpow2.def against the oracle.

The list is generated (tools/gen_nonpow2_kernels.py) and most of it was added without GPU time in round 1; here every curated
length runs, through the C ABI, in every role its kernels are registered for:
  ROWS        1-D C2C on contiguous lines (FP32 and FP64), forward and inverse, a batch that does not divide the CTA's tile;
              the fused even-length real transform of length 2N (R2C and C2R)
  COLS        the same length along the strided axis of a 2-D transform
  COLS+phase / ROWS_TOUT   a 1-D Four-Step of length N*N with the split forced to (N, N)
  B2_KD       DCT-II / DCT-III of that length on contiguous rows and along a strided axis
  B2_KB       Bluestein with that padded length (a prime just below M/2)
Tolerances: north-star 1e-6 (FP32) / 1e-12 (FP64) relative l2 against the double-precision oracle."""
import os
import re

import numpy as np
import pytest

import vkfft_oracle as orc

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _parse():
    rows, cols, tout, dct_rows, dct_cols, blue = {}, {}, {}, {}, {}, {}
    for line in open(os.path.join(ROOT, "vkfft_b200", "csrc", "kernel_list_nonpow2.def")):
        m = re.match(r"(B2_K[A-Z]*)\((.*)\)\s*(//.*)?$", line.strip())
        if not m:
            continue
        macro, args = m.group(1), [a.strip() for a in m.group(2).split(",")]
        if macro in ("B2_K", "B2_KD"):
            kind, typ, rad = args[1], args[2], [int(a) for a in args[7:]]
        elif macro == "B2_KB":
            kind, typ, rad = "ROWS", args[1], [int(a) for a in args[6:]]
        else:
            continue
        n = int(np.prod(rad))
        tgt = {("B2_K", "ROWS"): rows, ("B2_K", "COLS"): cols, ("B2_K", "ROWS_TOUT"): tout, ("B2_KD", "ROWS"): dct_rows,
               ("B2_KD", "COLS"): dct_cols, ("B2_KB", "ROWS"): blue}.get((macro, kind))
        if tgt is not None:
            tgt.setdefault(n, set()).add(typ)
    return rows, cols, tout, dct_rows, dct_cols, blue


ROWS, COLS, TOUT, DCT_ROWS, DCT_COLS, BLUE = _parse()


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


def _tol(double):
    return 1e-12 if double else 1e-6


def test_the_list_was_parsed():
    assert len(ROWS) > 150 and len(COLS) > 100 and len(DCT_ROWS) > 100 and len(BLUE) > 30


@pytest.mark.parametrize("n", sorted(ROWS))
def test_contiguous_lines_c2c_and_even_length_real(gpu, n):
    for typ in sorted(ROWS[n]):
        double = typ == "double"
        batch = 11
        x = orc.random_input((batch, n), np.complex128 if double else np.complex64, seed=n)
        for inv in (-1, 1):
            y = _run(gpu, x, inv, FFTdim=1, size=[n], numberBatches=batch, doublePrecision=int(double))
            assert orc.error_metrics(y, orc.c2c(x, 1, inv == 1))["l2_rel"] < _tol(double), (n, typ, inv)
        # the fused Hermitian pass: real transform of length 2n on the same kernel
        rdt, cdt = (np.float64, np.complex128) if double else (np.float32, np.complex64)
        r = orc.random_input((batch, 2 * n), rdt, seed=n + 1)
        buf = np.zeros((batch, 2 * n + 2), rdt)
        buf[:, :2 * n] = r
        y = _run(gpu, buf, -1, FFTdim=1, size=[2 * n], numberBatches=batch, performR2C=1, doublePrecision=int(double))
        assert orc.error_metrics(y.view(cdt), orc.r2c(r, 1))["l2_rel"] < _tol(double), (n, typ, "r2c")
        z = _run(gpu, y, 1, FFTdim=1, size=[2 * n], numberBatches=batch, performR2C=1, doublePrecision=int(double))
        assert orc.error_metrics(z[:, :2 * n], r.astype(np.float64) * 2 * n)["l2_rel"] < _tol(double), (n, typ, "c2r")


@pytest.mark.parametrize("n", sorted(COLS))
def test_strided_axis(gpu, n):
    for typ in sorted(COLS[n]):
        double = typ == "double"
        nx, batch = 40, 2                      # 40 neighbouring lines: not a multiple of the 8/16-line tiles
        x = orc.random_input((batch, n, nx), np.complex128 if double else np.complex64, seed=n + 2)
        for inv in (-1, 1):
            y = _run(gpu, x, inv, FFTdim=2, size=[nx, n], numberBatches=batch, doublePrecision=int(double))
            assert orc.error_metrics(y, orc.c2c(x, 2, inv == 1))["l2_rel"] < _tol(double), (n, typ, inv)


@pytest.mark.parametrize("n", sorted(set(TOUT) & set(COLS)))
def test_four_step_with_the_length_as_both_factors(gpu, n):
    if n * n > (1 << 24):
        pytest.skip("N*N beyond 2^24 points")
    old = os.environ.get("B200FFT_FOUR_STEP_SPLIT")
    os.environ["B200FFT_FOUR_STEP_SPLIT"] = f"{n},{n}"
    try:
        x = orc.random_input((2, n * n), np.complex64, seed=n + 3)
        for inv in (-1, 1):
            y = _run(gpu, x, inv, FFTdim=1, size=[n * n], numberBatches=2)
            assert orc.error_metrics(y, orc.c2c(x, 1, inv == 1))["l2_rel"] < 1e-6, (n, inv)
    finally:
        if old is None:
            os.environ.pop("B200FFT_FOUR_STEP_SPLIT", None)
        else:
            os.environ["B200FFT_FOUR_STEP_SPLIT"] = old


@pytest.mark.parametrize("n", sorted(set(DCT_ROWS) | set(DCT_COLS)))
def test_fused_dct23(gpu, n):
    from gpu_util import assert_f32_parity
    for kind in (2, 3):
        if n in DCT_ROWS:
            x = orc.random_input((7, n), np.float32, seed=n + kind)
            for inv in (-1, 1):
                y = _run(gpu, x, inv, FFTdim=1, size=[n], numberBatches=7, performDCT=kind)
                assert_f32_parity(y, orc.dct(x, kind, 1, inverse=(inv == 1)), x, (n,), 7, inv, perform_dct=kind)
        if n in DCT_COLS:
            x = orc.random_input((2, n, 36), np.float32, seed=n + kind + 5)
            for inv in (-1, 1):
                y = _run(gpu, x, inv, FFTdim=2, size=[36, n], numberBatches=2, performDCT=kind)
                assert_f32_parity(y, orc.dct(x, kind, 2, inverse=(inv == 1)), x, (36, n), 2, inv, perform_dct=kind)


def _prev_prime(m):
    def is_p(k):
        return k > 1 and all(k % d for d in range(2, int(k ** 0.5) + 1))
    while not is_p(m):
        m -= 1
    return m


@pytest.mark.parametrize("m", sorted(BLUE))
def test_bluestein_with_a_curated_padded_length(gpu, m):
    n = _prev_prime((m + 1) // 2)              # the largest prime whose 2N-1 still fits this padded length
    if n < 131:
        pytest.skip("primes up to 127 run as Rader stages")
    for typ in sorted(BLUE[m]):
        double = typ == "double"
        x = orc.random_input((5, n), np.complex128 if double else np.complex64, seed=m)
        for inv in (-1, 1):
            y = _run(gpu, x, inv, FFTdim=1, size=[n], numberBatches=5, doublePrecision=int(double))
            assert orc.error_metrics(y, orc.c2c(x, 1, inv == 1))["l2_rel"] < _tol(double), (m, n, typ, inv)
