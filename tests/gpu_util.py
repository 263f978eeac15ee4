"""Helpers for the -m gpu tests: run a plan through the C ABI (ctypes) on torch-owned device memory, and the stored results
of the unmodified reference's CUDA backend that the tests compare with."""
import hashlib
import os

import numpy as np

import vkfft_b200 as vk

# What the reference computed on the tests' inputs, recorded on a B200 from the reference built into oracle/_ref
# (oracle/Makefile): per case the reference's l2 error against the exact result and/or a sketch of its output (see sketch()).
# B200FFT_RECORD_REFERENCE=<file.npz> runs the reference for the cases this file does not hold yet and writes every case the
# tests asked for to <file.npz>:
#     B200FFT_RECORD_REFERENCE=$PWD/reference_gpu.npz python -m pytest -m gpu tests   (then copy it to REFERENCE_GOLDEN)
REFERENCE_GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_gpu", "cases.npz")
_RECORD = os.environ.get("B200FFT_RECORD_REFERENCE")
_golden = None        # {"sketch": {case: sketch}, "l2_exact": {case: l2}} read from REFERENCE_GOLDEN
_recorded = None      # the same for what a recording run writes
SKETCH_BUCKETS = 64


def _load_golden(path):
    if not os.path.exists(path):
        return {"sketch": {}, "l2_exact": {}}
    z = np.load(path)
    return {"sketch": dict(zip(z["sketch_keys"].astype(str), z["sketches"])),
            "l2_exact": dict(zip(z["l2_keys"].astype(str), z["l2_exact"].tolist()))}


def _save_golden(path, g):
    sk = sorted(g["sketch"])
    l2 = sorted(g["l2_exact"])
    np.savez_compressed(path, sketch_keys=np.array(sk, dtype="S"), sketches=np.array([g["sketch"][k] for k in sk], np.complex128).reshape(len(sk), SKETCH_BUCKETS),
                        l2_keys=np.array(l2, dtype="S"), l2_exact=np.array([g["l2_exact"][k] for k in l2], np.float64))


def sketch(a, k=SKETCH_BUCKETS):
    """CountSketch of `a` (k complex128 values): element i is added, with sign s(i), to bucket h(i); h and s are fixed by the
    array's size.  The sketch is linear, so sketch(a) - sketch(b) = sketch(a - b), and its l2 norm estimates ||a - b|| to about
    10 % with every element taking part -- which lets a few hundred bytes stand in for an output of any size."""
    a = np.asarray(a).astype(np.complex128).ravel()
    rng = np.random.default_rng(a.size)
    h = rng.integers(0, k, a.size)
    s = rng.integers(0, 2, a.size) * 2.0 - 1.0
    return np.bincount(h, s * a.real, k) + 1j * np.bincount(h, s * a.imag, k)


def sketch_l2_rel(sk_a, sk_ref):
    """l2_rel(a, ref) estimated from the sketches of a and ref"""
    return float(np.linalg.norm(sk_a - sk_ref) / max(np.linalg.norm(sk_ref), 1e-300))


def reference(x, size_xyz, batch, inverse, double=False, use_lut=1, exact=None, crop=None, sketched=True, **kw):
    """The reference's result for `x` through the plan (size_xyz, batch, double, use_lut, kw), direction `inverse`:
    {"sketch": sketch of its output (of output[..., :crop] when crop is given; when `sketched`), "l2_exact": its l2_rel
    against `exact` (when given)}.  Read from REFERENCE_GOLDEN; recorded when B200FFT_RECORD_REFERENCE is set."""
    global _golden, _recorded
    x = np.ascontiguousarray(x)
    key = (f"{','.join(map(str, size_xyz))} b{batch} {'f64' if double else 'f32'} inv{inverse} lut{use_lut} "
           + " ".join(f"{k}={v}" for k, v in sorted(kw.items())) + (f" crop{crop}" if crop else "") + f" x{x.dtype}{x.shape}:"
           + hashlib.sha1(x.tobytes()).hexdigest()[:12])
    want = (["sketch"] if sketched else []) + (["l2_exact"] if exact is not None else [])
    if _golden is None:
        _golden = _load_golden(REFERENCE_GOLDEN)
    if _RECORD:
        if _recorded is None:
            _recorded = {"sketch": {}, "l2_exact": {}}
        if not all(key in _golden[w] for w in want):
            import vkfft_oracle as orc
            torch = torch_mod()
            t = torch.from_numpy(x.copy()).cuda()
            rc = orc.ref_run(orc.ref_desc(size_xyz, batch, double, use_lut=use_lut, **kw), inverse, t.data_ptr())
            assert rc == 0, rc
            theirs = t.cpu().numpy()[..., :crop]
            _golden["sketch"][key] = sketch(theirs)
            if exact is not None:
                _golden["l2_exact"][key] = orc.error_metrics(theirs, exact)["l2_rel"]
        for w in want:
            _recorded[w][key] = _golden[w][key]
        _save_golden(_RECORD, _recorded)
    for w in want:
        assert key in _golden[w], f"no recorded reference {w} for {key} (see REFERENCE_GOLDEN)"
    return {w: _golden[w][key] for w in want}


def torch_mod():
    import torch
    return torch


def run_c2c(x_np, size_xyz, batches=1, inverse=-1, double=False, **cfgkw):
    """x_np: numpy complex array [batch, ..., y, x] (contiguous).  Returns the transformed numpy array."""
    torch = torch_mod()
    t = torch.from_numpy(np.ascontiguousarray(x_np)).cuda()
    cfg = vk.VkFFTConfiguration(FFTdim=len(size_xyz), size=list(size_xyz), numberBatches=batches, device=0,
                                doublePrecision=int(double), **cfgkw)
    app = vk.VkFFTApplication()
    rc = vk.initializeVkFFT(app, cfg)
    assert rc == vk.VKFFT_SUCCESS, vk.getVkFFTErrorString(rc)
    try:
        rc = vk.VkFFTAppend(app, inverse, vk.VkFFTLaunchParams(buffer=t))
        assert rc == vk.VKFFT_SUCCESS, vk.getVkFFTErrorString(rc)
        torch.cuda.synchronize()
        out = t.cpu().numpy()
    finally:
        vk.deleteVkFFT(app)
    return out


def assert_f32_parity(mine, exact, x, size_xyz, batch, inverse, tol=1e-6, **kw):
    """north_star tolerance for FP32: 1e-6 relative (l2) against the exact result.  Where a transform's own conditioning puts
    BOTH engines beyond that (the composed real transforms: the reference's FP32 error reaches ~1.4e-6, README.md:76-80),
    the criterion of the C2C reference test applies instead: this engine is at least as close to the exact result as the
    unmodified reference's CUDA backend on the same input x through the same plan (|mine - exact| <= 1.05 |reference - exact|)."""
    import vkfft_oracle as orc
    e_m = orc.error_metrics(mine, exact)["l2_rel"]
    if e_m < tol and not _RECORD:    # a recording run records every case, whatever this engine's error
        return e_m
    e_t = reference(x, size_xyz, batch, inverse, exact=exact, sketched=False, **kw)["l2_exact"]
    if e_m < tol:
        return e_m
    assert e_m <= 1.05 * e_t + 1e-8, f"l2_rel {e_m:.3e} vs reference {e_t:.3e} (north-star 1e-6)"
    return e_m
