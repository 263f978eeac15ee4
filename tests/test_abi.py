"""CPU: the C-ABI library loads, exports every symbol include/b200fft.h declares, the header-only vkFFT.h shim
compiles as C and C++ with the reference's struct layout, and host-side error behaviour matches the reference.
(No compute calls here: there is no GPU in the -m "not gpu" environment.)"""
import json
import os
import re
import subprocess
import sys
import tempfile

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# sizeof / offsetof of every member of the drop-in structs as the reference's own vkFFT.h (VkFFT 1.3.4, VKFFT_BACKEND=1)
# lays them out; written by `python tests/test_abi.py <reference>/vkFFT`
REFERENCE_LAYOUT = os.path.join(ROOT, "tests", "golden", "reference_vkfft_layout.json")


def test_library_exports_every_declared_symbol(built_lib):
    from vkfft_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "b200fft.h")).read()
    declared = set(re.findall(r"\b(b200fft_[a-z_]+)\s*\(", hdr))
    assert declared == set(_lib.EXPORTS), declared ^ set(_lib.EXPORTS)
    for s in declared:
        assert hasattr(built_lib, s), s
    assert built_lib.b200fft_kernel_count() > 100
    assert built_lib.b200fft_error_string(3002) == b"VKFFT_ERROR_UNSUPPORTED_FFT_LENGTH"


def test_desc_struct_layout_matches_header(built_lib):
    import ctypes
    from vkfft_b200 import _lib
    src = r'''
    #include "b200fft.h"
    #include <stdio.h>
    #include <stddef.h>
    int main(void){ printf("%zu %zu %zu %zu %zu\n", sizeof(b200fft_desc), offsetof(b200fft_desc, buffer_stride),
        offsetof(b200fft_desc, device), sizeof(b200fft_buffers), sizeof(b200fft_plan_info)); return 0; }'''
    with tempfile.TemporaryDirectory() as td:
        open(os.path.join(td, "t.c"), "w").write(src)
        subprocess.check_call(["gcc", "-std=c99", "-I", os.path.join(ROOT, "include"), os.path.join(td, "t.c"), "-o",
                               os.path.join(td, "t")])
        vals = list(map(int, subprocess.check_output([os.path.join(td, "t")]).split()))
    assert vals == [ctypes.sizeof(_lib.b200fft_desc), _lib.b200fft_desc.buffer_stride.offset,
                    _lib.b200fft_desc.device.offset, ctypes.sizeof(_lib.b200fft_buffers),
                    ctypes.sizeof(_lib.b200fft_plan_info)]


def _struct_members(header_text, struct_name):
    """member names of `typedef struct { ... } struct_name;` in declaration order (handles `a, *b, c[N]` lists)"""
    import re
    end = header_text.index("} " + struct_name + ";")
    start = header_text.rindex("typedef struct", 0, end)
    body = re.sub(r"/\*.*?\*/", "", header_text[start:end], flags=re.S)
    body = re.sub(r"//[^\n]*", "", body)
    names = []
    for decl in body[body.index("{") + 1:].split(";"):
        decl = decl.strip()
        if not decl or decl.startswith("#"):
            continue
        first, *rest = decl.split(",")
        parts = [first.split()[-1]] + rest if first.split() else rest
        for q in parts:
            q = q.strip().lstrip("*").strip()
            q = re.sub(r"\[.*", "", q)
            if re.fullmatch(r"[A-Za-z_][A-Za-z0-9_]*", q):
                names.append(q)
    return names


def _layout_dump(include_dirs, defines, members, lang):
    """compile AND RUN a probe printing sizeof + offsetof of every member; returns {name: value}"""
    cuda = "/usr/local/cuda"
    lines = ['#include "vkFFT.h"', "#include <stdio.h>", "#include <stddef.h>", "int main(void){",
             'printf("sizeof.VkFFTConfiguration %zu\\n", sizeof(VkFFTConfiguration));',
             'printf("sizeof.VkFFTLaunchParams %zu\\n", sizeof(VkFFTLaunchParams));']
    for st, ms in members.items():
        for m in ms:
            lines.append(f'printf("{st}.{m} %zu\\n", offsetof({st}, {m}));')
    lines.append("return 0; }")
    with tempfile.TemporaryDirectory() as td:
        ext = "c" if lang == "c" else "cpp"
        f = os.path.join(td, "t." + ext)
        open(f, "w").write("\n".join(lines))
        cc = ["gcc", "-std=c99"] if lang == "c" else ["g++", "-std=c++11"]
        cmd = cc + ["-w"] + [f"-D{d}" for d in defines]
        for d in include_dirs + [os.path.join(cuda, "include")]:
            cmd += ["-I", d]
        exe = os.path.join(td, "probe")
        # the probe only uses sizeof/offsetof: the header's forwarding functions are never referenced, nothing to link
        subprocess.check_call(cmd + [f, "-o", exe, "-Wl,--unresolved-symbols=ignore-all"])
        out = subprocess.run([exe], capture_output=True, text=True, check=True).stdout
    return {l.split()[0]: int(l.split()[1]) for l in out.strip().split("\n")}


@pytest.mark.parametrize("lang", ["c", "c++"])
def test_vkfft_shim_header_layout(lang):
    """sizeof/offsetof of the drop-in structs == the reference's VKFFT_BACKEND==1 build.  The probe is compiled, RUN and
    compared: against the known numbers of the reference headers (SURVEY.md section 7: VkFFTConfiguration 1168 B,
    VkFFTLaunchParams 80 B, buffer@152, numberBatches@272, doublePrecision@360, performR2C@408) and member by member against
    the same probe compiled from the reference's own header (REFERENCE_LAYOUT)."""
    cuda = "/usr/local/cuda"
    if not os.path.exists(os.path.join(cuda, "include", "cuda.h")):
        pytest.skip("CUDA headers not present")
    members = _shim_members()
    assert len(members["VkFFTConfiguration"]) > 100 and len(members["VkFFTLaunchParams"]) >= 9
    mine = _layout_dump([os.path.join(ROOT, "include")], ["VKFFT_BACKEND=1"], members, lang)
    assert mine["sizeof.VkFFTConfiguration"] == 1168 and mine["sizeof.VkFFTLaunchParams"] == 80
    assert mine["VkFFTConfiguration.buffer"] == 152 and mine["VkFFTConfiguration.numberBatches"] == 272
    assert mine["VkFFTConfiguration.doublePrecision"] == 360 and mine["VkFFTConfiguration.performR2C"] == 408
    theirs = json.load(open(REFERENCE_LAYOUT))
    assert mine == theirs, {k: (mine[k], theirs.get(k)) for k in mine if mine[k] != theirs.get(k)}


def _shim_members():
    hdr = open(os.path.join(ROOT, "include", "vkFFT.h")).read()
    return {"VkFFTConfiguration": _struct_members(hdr, "VkFFTConfiguration"),
            "VkFFTLaunchParams": _struct_members(hdr, "VkFFTLaunchParams")}


def test_python_api_host_side_errors(built_lib):
    import vkfft_b200 as vk
    app = vk.VkFFTApplication()
    assert vk.initializeVkFFT(None, vk.VkFFTConfiguration()) == vk.VKFFT_ERROR_EMPTY_app
    assert vk.initializeVkFFT(app, vk.VkFFTConfiguration(FFTdim=1, size=[8])) == vk.VKFFT_ERROR_INVALID_DEVICE
    assert vk.initializeVkFFT(app, vk.VkFFTConfiguration(FFTdim=0, size=[8], device=0)) == vk.VKFFT_ERROR_EMPTY_FFTdim
    assert vk.initializeVkFFT(app, vk.VkFFTConfiguration(FFTdim=5, size=[8], device=0)) == vk.VKFFT_ERROR_FFTdim_GT_MAX_FFT_DIMENSIONS
    assert vk.initializeVkFFT(app, vk.VkFFTConfiguration(FFTdim=1, size=[0], device=0)) == vk.VKFFT_ERROR_EMPTY_size
    assert vk.VkFFTAppend(app, -1, None) == vk.VKFFT_ERROR_PLAN_NOT_INITIALIZED
    assert vk.VkFFTGetVersion() == 10304
    # no GPU here: plan creation must fail loudly, never fall back to a CPU path
    import torch
    if not torch.cuda.is_available():
        assert vk.initializeVkFFT(app, vk.VkFFTConfiguration(FFTdim=1, size=[8], device=0)) == vk.VKFFT_ERROR_INVALID_DEVICE


def _build_sample(td):
    cuda = "/usr/local/cuda"
    exe = os.path.join(td, "drop_in_sample")
    subprocess.check_call(["g++", "-std=c++11", "-O1", os.path.join(ROOT, "tests", "cpp", "drop_in_sample.cpp"), "-o", exe,
                           "-I", os.path.join(ROOT, "include"), "-I", os.path.join(cuda, "include"),
                           "-L", os.path.join(ROOT, "vkfft_b200", "lib"), "-lb200fft",
                           "-L", os.path.join(cuda, "lib64"), "-L", os.path.join(cuda, "lib64", "stubs"), "-lcuda", "-lcudart",
                           "-Wl,-rpath," + os.path.join(ROOT, "vkfft_b200", "lib"), "-Wl,-rpath," + os.path.join(cuda, "lib64")])
    return exe


def test_reference_style_cpp_program_builds_against_the_shim(built_lib):
    if not os.path.exists("/usr/local/cuda/include/cuda.h"):
        pytest.skip("CUDA headers not present")
    with tempfile.TemporaryDirectory() as td:
        assert os.path.exists(_build_sample(td))


@pytest.mark.gpu
def test_reference_style_cpp_program_runs(built_lib):
    with tempfile.TemporaryDirectory() as td:
        out = subprocess.run([_build_sample(td)], capture_output=True, text=True)
        assert out.returncode == 0, out.stdout + out.stderr


def test_reference_testsuite_sources_build_against_the_shim(built_lib):
    """drop-in at source level: the reference's own VkFFT_TestSuite.cpp with its benchmark / convolution samples and utilities
    (unmodified, where they lie) compiles against include/vkFFT.h and links to libb200fft.so"""
    if not os.path.isdir("/root/reference/benchmark_scripts"):
        pytest.skip("reference tree not present")
    exe = os.path.join(ROOT, "oracle", "_ref", "VkFFT_TestSuite_b200")
    if os.path.exists(exe):
        os.unlink(exe)
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle"), "testsuite"], stdout=subprocess.DEVNULL)
    assert os.path.exists(exe)
    syms = subprocess.run(["nm", "-D", "--undefined-only", exe], capture_output=True, text=True).stdout
    for s in ("b200fft_plan_create", "b200fft_exec", "b200fft_plan_destroy", "b200fft_plan_axis_uploads"):
        assert s in syms, s                      # the samples' initializeVkFFT / VkFFTAppend / deleteVkFFT end in the C ABI
    assert "nvrtcCompileProgram" not in syms     # nothing is JIT-compiled any more


if __name__ == "__main__":
    # regenerate REFERENCE_LAYOUT from the directory holding the reference's vkFFT.h
    with open(REFERENCE_LAYOUT, "w") as f:
        json.dump(_layout_dump([sys.argv[1]], ["VKFFT_BACKEND=1"], _shim_members(), "c++"), f, indent=0, sort_keys=True)
        f.write("\n")
