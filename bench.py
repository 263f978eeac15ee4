#!/usr/bin/env python3
"""Benchmark of the hot path: BASELINE.json's metric on BASELINE.json's config[1].

  metric   batched 1-D C2C FP32 throughput in GFLOP/s (5 N log2 N per transform) + HBM roofline fraction
  workload the reference's sample_0 sweep (benchmark_scripts/vkFFT_scripts/src/sample_0_benchmark_VkFFT_single.cpp)
           at BASELINE's sizes: N = 2^7 .. 2^22, batch = 2^28 / N (one 2 GiB complex64 buffer per GPU), in place.
  step     one pass over the sweep: for every N one forward and one inverse transform of the whole buffer
           (32 transforms, 128 GiB of algorithmic HBM traffic per GPU per step).
  value    whole-job GFLOP/s with the buffer resident in HBM (CUDA events, max over ranks).
  e2e      the same step through the public API with HOST buffers: pinned-host -> HBM copy of the step's input,
           the sweep, and the HBM -> host read of the result, all inside the timed region.
  roofline the dominant kernel = the kernel with the LARGEST SHARE of the step's device time (per-launch CUDA events
           through b200fft_debug_exec_timed, aggregated by kernel over the sweep): algorithmic bytes per launch / mean
           launch time / measured peak; `kernel_shares` lists the top kernels, `step_frac` is the whole step.
  other_lengths  lengths off the power-of-two sweep (curated kernels, templates instantiated at plan time, Bluestein): ms per
              pair of ~512 MiB, roofline fraction, plan time, and the reference's CUDA backend beside it
  per_config  BASELINE configs 3-5 on one GPU (3-D FP64 256^3 / 512^3, 2-D R2C 4096^2, DCT-II 8192^2, 1-D 2^26): ms per
           forward+inverse pair, roofline fraction, and the unmodified reference's CUDA backend on the same GPU.
  sample0  the reference's own sample_0 benchmark binary (VkFFT_TestSuite -vkfft 0, "Benchmark score VkFFT") built from the
           reference's sources against this engine (oracle/_ref/VkFFT_TestSuite_b200) and against stock VkFFT
           (oracle/_ref/VkFFT_TestSuite_ref), both run here.
  dist_2p26  (N >= 2 GPUs) config 5: one 2^26-point sequence over all ranks, exchange fused into the FFT launches.
  cpu_baseline  pocketfft (scipy.fft) on the box's host cores, bounded sample -- stand-in for the reference's
           FFTW precision-test path (FFTW is not installed in this image).  Reported, not a target.
  vkfft_cuda_ref  the UNMODIFIED reference (CUDA backend, oracle/_ref) timed on the same GPU in the same run.

Launch:  python bench.py --gpus 1 --steps K --warmup W          (N>1: via torch.distributed.run, one rank per GPU)
         python bench.py --impl reference ...                   (the reference arm: CPU implementation of the path)
         python bench.py ... --dump-outputs DIR                 (also write what the last timed step computed, see dump_outputs)
"""
import argparse
import ctypes
import json
import math
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# torchrun exports OMP_NUM_THREADS=1, which also throttles pocketfft's worker pool: the CPU legs are meant to use
# every host core, so drop the cap before numpy/scipy are imported.
os.environ.pop("OMP_NUM_THREADS", None)

LOG2_MIN, LOG2_MAX = 7, 22
TOTAL_LOG2 = 28                      # 2^28 complex64 = 2 GiB
CPU_SAMPLE_LOG2 = 26                 # bounded sample for the CPU legs: 2^26 points (512 MiB) per N


def sizes():
    return [1 << k for k in range(LOG2_MIN, LOG2_MAX + 1)]


def flops_pair(n, points):
    """forward + inverse over `points` complex points organised as sequences of length n"""
    return 2 * 5.0 * points * math.log2(n)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "MEASURED_PEAKS.json (driver-measured copy bandwidth)"
        except Exception:
            pass
    return 6650.0, "fallback from B200_PROFILING.md (MEASURED_PEAKS.json absent)"


class ClockSampler:
    """samples nvidia-smi SM clocks + throttle reasons while the timed region runs"""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.idx)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------------------------
def cpu_sweep_once(np, sfft, bufs, workers):
    for n, a in bufs:
        y = sfft.fft(a, axis=1, workers=workers, overwrite_x=False)
        sfft.ifft(y, axis=1, workers=workers, overwrite_x=True, norm="forward")


def cpu_baseline(steps=1, warmup=0):
    """pocketfft, complex64, all host cores, the same sweep on a bounded sample (2^24 points per N)"""
    import numpy as np
    import scipy.fft as sfft
    cores = os.cpu_count() or 1
    rng = np.random.default_rng(0)
    pts = 1 << CPU_SAMPLE_LOG2
    base = (rng.uniform(-1, 1, pts).astype(np.float32) + 1j * rng.uniform(-1, 1, pts).astype(np.float32)).astype(np.complex64)
    bufs = [(n, base.reshape(pts // n, n)) for n in sizes()]
    fl = sum(flops_pair(n, pts) for n in sizes())
    for _ in range(warmup):
        cpu_sweep_once(np, sfft, bufs, cores)
    t0 = time.perf_counter()
    for _ in range(steps):
        cpu_sweep_once(np, sfft, bufs, cores)
    dt = (time.perf_counter() - t0) / steps
    return {"value": fl / dt / 1e9, "unit": "GFLOP/s", "cores": cores, "kind": "port",
            "sample": f"same sweep N=2^{LOG2_MIN}..2^{LOG2_MAX} fwd+inv, 2^{CPU_SAMPLE_LOG2} complex64 points per N "
                      f"(512 MiB instead of 2 GiB), scipy.fft/pocketfft workers={cores}; stand-in for the reference's "
                      "FFTW precision-test path (FFTW not installed)",
            "seconds_per_step": dt}, dt


def vkfft_cuda_reference(torch, buf, ns, iters=5, warm=2):
    """time the unmodified reference's CUDA backend (oracle/_ref) on the same buffer: ms per FFT+iFFT pair per N"""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import vkfft_oracle as orc
    if not orc.ref_available():
        return {"unavailable": "oracle/_ref/libvkfft_ref.so not built"}
    L = orc.ref_lib()
    out = {"per_n": {}, "impl": "DTolm/VkFFT 1.3.4 CUDA backend (NVRTC), unmodified, same GPU, same buffer",
           "warmup_pairs": warm, "timed_pairs": iters}
    total_ms, total_fl = 0.0, 0.0
    pts = buf.numel()
    score_terms = []
    for n in ns:
        d = orc.ref_desc((n,), pts // n, False, device=torch.cuda.current_device())
        h = ctypes.c_void_p()
        rc = L.vkref_open(ctypes.byref(d), ctypes.byref(h))
        if rc != 0:
            out["per_n"][str(n)] = {"error": rc}
            continue
        ms_e, ms_w = ctypes.c_double(), ctypes.c_double()
        rc = L.vkref_bench_pairs(h, buf.data_ptr(), warm, iters, ctypes.byref(ms_e), ctypes.byref(ms_w))
        up = L.vkref_axis0_uploads(h)
        L.vkref_close(h)
        buf.zero_()                      # unnormalised pairs overflow; reset (timing is data independent)
        if rc != 0:
            out["per_n"][str(n)] = {"error": rc}
            continue
        out["per_n"][str(n)] = {"ms_pair": round(ms_e.value, 4), "uploads": up}
        total_ms += ms_e.value
        total_fl += flops_pair(n, pts)
        score_terms.append((pts * 8 / 1024.0) / ms_e.value)      # sample_0: bufferSize_KB / ms per FFT+iFFT
    if total_ms > 0:
        out["gflops_sweep"] = total_fl / (total_ms * 1e-3) / 1e9
        out["ms_sweep"] = total_ms
        out["sample0_style_score"] = sum(score_terms) / len(score_terms)
    return out



DUMP_POINTS = 1 << 17                # points of the buffer written per array by --dump-outputs (1 MiB of complex64)


def dump_outputs(out_dir, torch, vk, apps, lp, buf, start, steps, sweep):
    """--dump-outputs: what the timed steps' last step computed, as a caller of each VkFFTAppend receives it in `buf`, written
    as DIR/<name>.npy float32 arrays [DUMP_POINTS, 2] (re, im) at one fixed, seeded sample of buffer positions:
      input                the buffer as the last step received it
      forward_n<N>, inverse_n<N>   the buffer after that step's forward / inverse transform of length N (in sweep order)
    The step is replayed from `start` (a copy of the buffer taken just before the timed steps) after the same number of sweeps;
    the replay must reproduce the timed steps' result bit for bit at the sampled positions, or nothing is written."""
    import numpy as np
    idx = np.sort(np.random.default_rng(0).choice(buf.numel(), DUMP_POINTS, replace=False))
    idx = torch.from_numpy(idx).to(buf.device)
    timed = buf[idx]
    buf.copy_(start)
    for _ in range(steps - 1):
        sweep()
    arrays = {"input": buf[idx]}
    for n, app, _ in apps:
        for inv, name in ((-1, "forward"), (1, "inverse")):
            rc = vk.VkFFTAppend(app, inv, lp)
            if rc:
                raise RuntimeError(vk.getVkFFTErrorString(rc))
            arrays[f"{name}_n{n}"] = buf[idx]
    assert torch.equal(buf[idx], timed), "the replayed step differs from the timed one"
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), torch.view_as_real(a).cpu().numpy())
    return {"dir": out_dir, "arrays": len(arrays), "points_per_array": DUMP_POINTS, "dtype": "float32 (re, im)"}


# ------------------------------------------------------------------------------------------------------------------
def bind_to_gpu_numa_node(local_rank):
    """Pin this rank's threads to the CPUs next to its GPU BEFORE the pinned host buffer is allocated (first touch puts the
    pages on that NUMA node): 8 ranks copying 4 GiB per step each otherwise meet on one socket's memory controllers."""
    try:
        bus = subprocess.run(["nvidia-smi", "--query-gpu=pci.bus_id", "--format=csv,noheader", "-i", str(local_rank)],
                             capture_output=True, text=True, timeout=20).stdout.strip().lower()
        if bus.startswith("00000000:"):
            bus = "0000:" + bus[len("00000000:"):]
        base = f"/sys/bus/pci/devices/{bus}"
        cpus = open(base + "/local_cpulist").read().strip()
        node = open(base + "/numa_node").read().strip()
        ids = set()
        for part in cpus.split(","):
            a, _, b = part.partition("-")
            ids.update(range(int(a), int(b or a) + 1))
        if ids:
            os.sched_setaffinity(0, ids)
            return {"numa_node": int(node), "cpus": cpus}
    except Exception as e:
        return {"error": repr(e)}
    return {"error": "no local_cpulist"}


def launch_labels(describe_text):
    """plan_describe lines -> one label per actual launch (a fused pair is one launch)"""
    import re
    out = []
    for l in describe_text.strip().split("\n"):
        if "runs inside the previous launch" in l:
            continue
        m = re.search(r"fused with the next launch: (FUSED4<[^\]]*?>),", l)
        if m:
            out.append(m.group(1))
            continue
        m = re.search(r" n=(\d+) (\S+)\[", l)
        what = l.split(": ", 1)[1].split(" n=")[0] if ": " in l else ""
        out.append(f"{m.group(2)} n={m.group(1)} ({what})" if m else l[:80])
    return out


def timed_launches(vk, app, inv, buffers, reps=3):
    """per-launch device times of one execution (CUDA events around every launch): [ms, ...], best of `reps`"""
    from vkfft_b200 import _lib
    L = _lib.load()
    L.b200fft_debug_exec_timed.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                           ctypes.c_int, ctypes.c_void_p]
    b = _lib.b200fft_buffers()
    b.buffer = buffers["buffer"]
    if buffers.get("temp"):
        b.temp_buffer = buffers["temp"]
    ms, kind, n = (ctypes.c_float * 64)(), (ctypes.c_int * 64)(), ctypes.c_int(0)
    best = None
    for _ in range(reps):
        rc = L.b200fft_debug_exec_timed(app._plan, inv, ctypes.byref(b), ms, kind, 64, ctypes.byref(n))
        if rc != 0:
            raise RuntimeError(vk.getVkFFTErrorString(rc))
        cur = [ms[i] for i in range(n.value) if kind[i] == 1]
        best = cur if best is None else [min(a, c) for a, c in zip(best, cur)]
    return best


CONFIG_CASES = [
    # BASELINE.json configs[2..4], single-GPU part: name, size_xyz, batch, double, engine kwargs, reference kwargs, real?
    ("config3: 3D C2C FP64 256^3 x8", (256, 256, 256), 8, True, {}, {}, False),
    ("config3: 3D C2C FP64 512^3 x1", (512, 512, 512), 1, True, {}, {}, False),
    ("config4: 2D R2C/C2R FP32 4096^2 x16", (4096, 4096), 16, False, dict(performR2C=1), dict(perform_r2c=1), True),
    ("config4: 2D DCT-II/III FP32 8192^2 x2", (8192, 8192), 2, False, dict(performDCT=2), dict(perform_dct=2), True),
    ("config5 (one GPU): 1D C2C FP32 2^26 x4", (1 << 26,), 4, False, {}, {}, False),
]


OTHER_LENGTHS = [
    # lengths off the power-of-two sweep, 1-D C2C FP32, ~512 MiB per transform: (N, which kind of kernel serves it)
    (1000, "curated ahead-of-time kernel"), (2187, "curated ahead-of-time kernel (3^7)"), (1088, "curated, direct radix-17 butterfly"),
    (1100, "template instantiated at plan time"), (2002, "template instantiated at plan time"), (34, "template instantiated at plan time (17 x 2)"),
    (127, "Bluestein in one launch"), (509, "Bluestein in one launch"), (1019, "Bluestein in one launch"), (4093, "Bluestein, two launches"),
    # halfPrecision = 1: the same number of points in half-precision storage (256 MiB per transform), FP32 arithmetic
    (-4096, "half-precision storage, plan-time variant of the tuned 4096-point kernel"),
    (-(1 << 20), "half-precision storage, Four-Step (factors up to 512, scratch in half as well)"),
]


def bench_other_lengths(torch, vk, peak, dev, warm=2, reps=5):
    """non power-of-two lengths: engine vs the unmodified reference's CUDA backend (which generates a kernel per plan)"""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import vkfft_oracle as orc
    rows = []
    for n, what in OTHER_LENGTHS:
        half = n < 0
        n = abs(n)
        batch = max(1, (1 << 26) // n)
        if half:
            buf = torch.zeros(batch * n, dtype=torch.int32, device=dev)       # (half re, half im) per element, all zero
        else:
            buf = torch.zeros(batch * n, dtype=torch.complex64, device=dev)
            torch.view_as_real(buf).uniform_(-1, 1)
        row = {"n": n, "batch": batch, "served_by": what}
        app = vk.VkFFTApplication()
        t0 = time.time()
        rc = vk.initializeVkFFT(app, vk.VkFFTConfiguration(FFTdim=1, size=[n], numberBatches=batch, device=dev.index, normalize=1, halfPrecision=int(half)))
        row["plan_seconds"] = round(time.time() - t0, 2)
        if rc != 0:
            row["error"] = vk.getVkFFTErrorString(rc)
        else:
            info = vk.planInfo(app)
            lp = vk.VkFFTLaunchParams(buffer=buf)
            for _ in range(warm):
                vk.VkFFTAppend(app, -1, lp); vk.VkFFTAppend(app, 1, lp)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(reps):
                vk.VkFFTAppend(app, -1, lp); vk.VkFFTAppend(app, 1, lp)
            b.record(); torch.cuda.synchronize()
            ms = a.elapsed_time(b) / reps
            alg = 4 * buf.numel() * (4 if half else 8)      # one read + one write of the lines per direction
            row.update(ms_pair=round(ms, 4), launches_forward=len(launch_labels(info["forward"])), frac_of_peak=round(alg / (ms * 1e-3) / 1e9 / peak, 4))
            vk.deleteVkFFT(app)
        if orc.ref_available() and not half:
            L = orc.ref_lib()
            d = orc.ref_desc((n,), batch, False, device=dev.index)
            h = ctypes.c_void_p()
            if L.vkref_open(ctypes.byref(d), ctypes.byref(h)) == 0:
                e, w = ctypes.c_double(), ctypes.c_double()
                buf.uniform_(-1e-3, 1e-3) if False else None
                if L.vkref_bench_pairs(h, buf.data_ptr(), warm, reps, ctypes.byref(e), ctypes.byref(w)) == 0:
                    row["reference_ms_pair"] = round(e.value, 4)
                L.vkref_close(h)
        rows.append(row)
        del buf
        torch.cuda.empty_cache()
    return rows


def bench_configs(torch, vk, peak, dev, warm=2, reps=5):
    """BASELINE configs 3-5 on this GPU: engine vs the unmodified reference's CUDA backend, same buffer, same warm-up/reps"""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import vkfft_oracle as orc
    rows = []
    for name, size, batch, dbl, kw, rkw, real in CONFIG_CASES:
        pts = batch
        for s_ in size:
            pts *= s_
        if kw.get("performR2C"):
            alloc = batch * (size[0] // 2 + 1) * 2
            for s_ in size[1:]:
                alloc *= s_
        else:
            alloc = pts * (1 if real else 2)
        buf = torch.zeros(alloc, dtype=torch.float64 if dbl else torch.float32, device=dev).uniform_(-1, 1)
        row = {"case": name}
        app = vk.VkFFTApplication()
        rc = vk.initializeVkFFT(app, vk.VkFFTConfiguration(FFTdim=len(size), size=list(size), numberBatches=batch, device=dev.index,
                                                           doublePrecision=int(dbl), normalize=1, **kw))
        if rc != 0:
            row["error"] = vk.getVkFFTErrorString(rc)
        else:
            info = vk.planInfo(app)
            lp = vk.VkFFTLaunchParams(buffer=buf)
            for _ in range(warm):
                vk.VkFFTAppend(app, -1, lp); vk.VkFFTAppend(app, 1, lp)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(reps):
                vk.VkFFTAppend(app, -1, lp); vk.VkFFTAppend(app, 1, lp)
            b.record(); torch.cuda.synchronize()
            ms = a.elapsed_time(b) / reps
            alg = 2 * info["algorithmic_bytes"]       # one read + one write of the data per transformed axis, both directions
            row.update(ms_pair=round(ms, 4), launches_forward=len(launch_labels(info["forward"])),
                       algorithmic_gb_pair=round(alg / 1e9, 3), frac_of_peak=round(alg / (ms * 1e-3) / 1e9 / peak, 4))
            vk.deleteVkFFT(app)
        if orc.ref_available():
            L = orc.ref_lib()
            d = orc.ref_desc(size, batch, dbl, device=dev.index, **rkw)
            h = ctypes.c_void_p()
            rc = L.vkref_open(ctypes.byref(d), ctypes.byref(h))
            if rc == 0:
                e, w = ctypes.c_double(), ctypes.c_double()
                buf.uniform_(-1e-3, 1e-3)
                rc = L.vkref_bench_pairs(h, buf.data_ptr(), warm, reps, ctypes.byref(e), ctypes.byref(w))
                row["reference_ms_pair"] = round(e.value, 4) if rc == 0 else f"error {rc}"
                L.vkref_close(h)
            else:
                row["reference_ms_pair"] = f"init error {rc}"
        rows.append(row)
        del buf
        torch.cuda.empty_cache()
    return rows


def sample0_scores(device_index):
    """the reference's sample_0 benchmark binary (VkFFT_TestSuite -vkfft 0), once linked to this engine and once stock"""
    import re
    out = {"formula": "mean over N = 2^3..2^27 (1 GiB buffer) of buffer_KB / ms per FFT+iFFT "
                      "(sample_0_benchmark_VkFFT_single.cpp:239-276)"}
    for key, exe in (("b200fft", "VkFFT_TestSuite_b200"), ("reference_vkfft_cuda", "VkFFT_TestSuite_ref")):
        path = os.path.join(ROOT, "oracle", "_ref", exe)
        if not os.path.exists(path):
            out[key] = {"unavailable": f"oracle/_ref/{exe} not built"}
            continue
        try:
            t0 = time.time()
            with tempfile.TemporaryDirectory() as td:      # the program writes its kernel cache to its working directory
                r = subprocess.run([path, "-d", str(device_index), "-vkfft", "0"], capture_output=True, text=True, timeout=900,
                                   cwd=td)
            m = re.search(r"Benchmark score VkFFT: (\d+)", r.stdout)
            per = {mm.group(1): float(mm.group(2)) for mm in re.finditer(r"VkFFT System: (\d+) .*?avg_time_per_step: ([0-9.]+) ms", r.stdout)}
            out[key] = {"score": int(m.group(1)) if m else None, "rc": r.returncode, "seconds": round(time.time() - t0, 1),
                        "ms_per_pair_by_log2n": per}
            if not m:
                out[key]["tail"] = (r.stdout + r.stderr)[-400:]
        except Exception as e:
            out[key] = {"error": repr(e)}
    return out


def bench_dist_2p26(torch, dist, vk, local_rank, rank, world):
    """config 5: ONE 2^26-point sequence over all ranks; the exchange is the peer loads/stores of the FFT launches"""
    from vkfft_b200.dist import FusedDistributedFFT1D
    n = 1 << 26
    dev = torch.device("cuda", local_rank)
    rec = {"n": "2^26", "world": world}
    f = FusedDistributedFFT1D(n, dist, local_rank, normalize=True)
    g = torch.Generator(device=dev).manual_seed(99)
    torch.view_as_real(f.local).uniform_(-1, 1, generator=g)
    x0 = f.local.clone()

    def pair():
        f(inverse=False); f(inverse=True)
    for _ in range(3):
        pair()
    dist.barrier(); torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 10
    a.record()
    for _ in range(reps):
        pair()
    b.record(); torch.cuda.synchronize()
    t = torch.tensor([a.elapsed_time(b) / reps / 2], device=dev, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    f.check()
    err = (f.local - x0).abs().double().norm() / x0.abs().double().norm()
    e = torch.tensor([float(err)], device=dev, dtype=torch.float64)
    dist.all_reduce(e, op=dist.ReduceOp.MAX)
    dist.barrier()
    f.timed(False)
    br = f.timed(False)
    rec.update(fused_ms_per_transform=round(t.item(), 4), gflops=round(5 * n * 26 / (t.item() * 1e-3) / 1e9, 1),
               roundtrip_rel_err_after_26_transforms=e.item(), launches_rank0=[(k, round(m, 4)) for k, m in br],
               nvlink_bytes_per_gpu_per_direction=int(n * 8 / world * (world - 1) / world) * 2,
               note="bytes: launch 1 gathers (R-1)/R of its columns and scatters (R-1)/R of its results, the last launch scatters again")
    f.close()
    dist.barrier()
    if rank == 0:
        # the same transform on one GPU, for the speed-up
        buf = torch.zeros(n, dtype=torch.complex64, device=dev)
        app = vk.VkFFTApplication()
        if vk.initializeVkFFT(app, vk.VkFFTConfiguration(FFTdim=1, size=[n], device=local_rank, normalize=1)) == 0:
            lp = vk.VkFFTLaunchParams(buffer=buf)
            for _ in range(3):
                vk.VkFFTAppend(app, -1, lp); vk.VkFFTAppend(app, 1, lp)
            a.record()
            for _ in range(reps):
                vk.VkFFTAppend(app, -1, lp); vk.VkFFTAppend(app, 1, lp)
            b.record(); torch.cuda.synchronize()
            rec["single_gpu_ms_per_transform"] = round(a.elapsed_time(b) / reps / 2, 4)
            rec["speedup_vs_one_gpu"] = round(rec["single_gpu_ms_per_transform"] / rec["fused_ms_per_transform"], 3)
            vk.deleteVkFFT(app)
        del buf
    dist.barrier()
    return rec


# ------------------------------------------------------------------------------------------------------------------
def run_reference_arm(args, rank, world):
    """--impl reference: the reference's CPU implementation of the path (its FFTW precision-test path; pocketfft
    stand-in) on the box's host cores, same metric/config, bounded sample.  Rank 0 only."""
    if rank != 0:
        return
    cb, dt = cpu_baseline(steps=max(1, args.steps), warmup=args.warmup)
    line = {
        "impl": "reference", "metric": "batched 1D C2C FP32 throughput (sample_0 sweep N=2^7..2^22, fwd+inv)",
        "value": cb["value"], "unit": "GFLOP/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": "sample_0 sweep N=2^7..2^22 C2C FP32 fwd+inv", "sample_points_per_n": 1 << CPU_SAMPLE_LOG2,
                   "note": "reference has no CPU FFT of its own; its CPU path is FFTW (absent) -> pocketfft stand-in"},
        "cpu_baseline": cb,
        "e2e": {"value": cb["value"], "unit": "GFLOP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    if not args.no_ref_gpu:
        try:
            import torch
            if torch.cuda.is_available():
                buf = torch.zeros(1 << TOTAL_LOG2, dtype=torch.complex64, device="cuda")
                line["vkfft_cuda_ref"] = vkfft_cuda_reference(torch, buf, sizes())
        except Exception as e:  # the CPU arm stands on its own
            line["vkfft_cuda_ref"] = {"unavailable": repr(e)}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-ref-gpu", action="store_true", help="skip timing the reference's CUDA backend")
    ap.add_argument("--no-cpu", action="store_true", help="skip the CPU baseline leg")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--no-configs", action="store_true", help="skip the BASELINE config 3-5 legs")
    ap.add_argument("--no-sample0", action="store_true", help="skip the reference's sample_0 benchmark binaries")
    ap.add_argument("--no-dist", action="store_true", help="skip the distributed 2^26 record (N >= 2)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed to DIR/*.npy (rank 0)")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return

    numa = bind_to_gpu_numa_node(local_rank)
    import torch
    import vkfft_b200 as vk
    assert torch.cuda.is_available(), "bench.py needs a GPU (there is no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    dev = torch.device("cuda", local_rank)
    pts = 1 << TOTAL_LOG2
    ns = sizes()
    buf = torch.empty(pts, dtype=torch.complex64, device=dev)
    tmp = torch.empty(pts, dtype=torch.complex64, device=dev)
    g = torch.Generator(device=dev).manual_seed(1234 + rank)
    torch.view_as_real(buf).uniform_(-1, 1, generator=g)
    stream = torch.cuda.current_stream().cuda_stream

    apps, launches_per_step = [], 0
    for n in ns:
        app = vk.VkFFTApplication()
        rc = vk.initializeVkFFT(app, vk.VkFFTConfiguration(FFTdim=1, size=[n], numberBatches=pts // n, device=local_rank,
                                                           normalize=1, userTempBuffer=1, tempBufferSize=pts * 8))
        assert rc == 0, (n, vk.getVkFFTErrorString(rc))
        info = vk.planInfo(app)
        launches_per_step += info["num_passes_forward"] + info["num_passes_inverse"]
        apps.append((n, app, info))
    lp = vk.VkFFTLaunchParams(buffer=buf, tempBuffer=tmp, stream=stream)

    def sweep():
        for n, app, _ in apps:
            rc = vk.VkFFTAppend(app, -1, lp)
            rc |= vk.VkFFTAppend(app, 1, lp)
            if rc:
                raise RuntimeError(vk.getVkFFTErrorString(rc))

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- value: inputs resident in HBM ---------------------------------------------------------------------
    for _ in range(args.warmup):
        sweep()
    barrier()
    start = buf.clone() if args.dump_outputs and rank == 0 else None
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        sweep()
    e1.record()
    barrier()
    ms_total = e0.elapsed_time(e1)
    clocks = sampler.stop() if rank == 0 else None
    ms_step = ms_total / args.steps
    if dist is not None:
        t = torch.tensor([ms_step], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_step = float(t.item())
    fl_step = sum(flops_pair(n, pts) for n in ns)
    value = world * fl_step / (ms_step * 1e-3) / 1e9
    dumped = None
    if start is not None:
        dumped = dump_outputs(args.dump_outputs, torch, vk, apps, lp, buf, start, args.steps, sweep)
        del start
        torch.cuda.empty_cache()

    # ---- per-N breakdown (rank 0 reports) ---------------------------------------------------------------------------
    peak, peak_src = measured_peaks()
    per_n = {}
    alg_bytes_dir = 2 * 8 * pts      # one read + one write of every complex64 point, per direction
    for n, app, info in apps:
        reps = 5
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for _ in range(2):
            vk.VkFFTAppend(app, -1, lp); vk.VkFFTAppend(app, 1, lp)
        a.record()
        for _ in range(reps):
            vk.VkFFTAppend(app, -1, lp); vk.VkFFTAppend(app, 1, lp)
        b.record()
        torch.cuda.synchronize()
        ms_pair = a.elapsed_time(b) / reps
        gbs = 2 * alg_bytes_dir / (ms_pair * 1e-3) / 1e9
        per_n[str(n)] = {"ms_pair": round(ms_pair, 4), "gflops": round(flops_pair(n, pts) / (ms_pair * 1e-3) / 1e9, 1),
                         "alg_gbs": round(gbs, 1), "frac_of_peak": round(gbs / peak, 4),
                         "launches": len(launch_labels(info["forward"]))}
    # ---- which kernel dominates the step?  One execution of every plan with CUDA events around every launch, aggregated by
    # kernel over the whole sweep (both directions).  The roofline line is about THAT kernel; every launch of the sweep reads
    # and writes the 2 GiB buffer exactly once (a fused Four-Step launch included), so algorithmic bytes per launch are equal.
    shares = {}
    if rank == 0:
        for n, app, info in apps:
            for inv, key in ((-1, "forward"), (1, "inverse")):
                labels = launch_labels(info[key])
                times = timed_launches(vk, app, inv, {"buffer": buf.data_ptr(), "temp": tmp.data_ptr()})
                for lab, t in zip(labels, times):
                    if lab.startswith("FUSED4") or "init" in lab:
                        pass
                    e = shares.setdefault(lab.split(" (")[0], {"ms": 0.0, "launches": 0})
                    e["ms"] += t; e["launches"] += 1
    tot_ms = sum(e["ms"] for e in shares.values()) or 1.0
    ranked = sorted(shares.items(), key=lambda kv: -kv[1]["ms"])
    kernel_shares = [{"kernel": k, "share_of_step": round(e["ms"] / tot_ms, 4), "launches_per_step": e["launches"],
                      "ms_per_launch": round(e["ms"] / e["launches"], 4),
                      "frac_of_peak": round(alg_bytes_dir / (e["ms"] / e["launches"] * 1e-3) / 1e9 / peak, 4)} for k, e in ranked[:8]]
    roofline = {"bound": "hbm", "peak": peak, "unit": "GB/s", "peak_source": peak_src, "traffic": None,
                "step_frac": round((len(ns) * 2 * alg_bytes_dir) / (ms_step * 1e-3) / 1e9 / peak, 4),
                "algorithmic_bytes_per_launch": alg_bytes_dir}
    if ranked:
        k, e = ranked[0]
        ms_dom = e["ms"] / e["launches"]
        ach = alg_bytes_dir / (ms_dom * 1e-3) / 1e9
        roofline.update(kernel=k, share_of_step=round(e["ms"] / tot_ms, 4), achieved=round(ach, 1), frac=round(ach / peak, 4),
                        ms_per_launch=round(ms_dom, 4), launches_per_step=e["launches"],
                        how="largest share of the step's device time; per-launch CUDA events on the launch stream "
                            "(b200fft_debug_exec_timed), mean over its launches in the sweep")
        tr = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tr):
            try:
                for rec in json.load(open(tr)):
                    if rec["kernel"] in k or k in rec["kernel"]:
                        roofline["traffic"] = rec["dram_bytes_per_launch"]
                        roofline["traffic_source"] = rec.get("source")
            except Exception:
                pass

    # restore a sane buffer and verify the round trip the bench has been doing (normalize=1 -> identity)
    torch.view_as_real(buf).uniform_(-1, 1, generator=g)
    ref0 = buf[: 1 << 20].clone()
    sweep()
    torch.cuda.synchronize()
    rt_err = float((buf[: 1 << 20] - ref0).abs().double().norm() / ref0.abs().double().norm())

    # ---- e2e: host buffers, copies inside the timed region ------------------------------------------------------
    host = torch.empty(pts, dtype=torch.complex64, pin_memory=True)
    torch.view_as_real(host).uniform_(-1, 1)
    nbytes = pts * 8

    # The batch is cut into chunks that travel through three streams: while chunk c is being transformed, chunk c+1 is on
    # its way in and chunk c-1 on its way out (PCIe is full duplex), all through VkFFTAppend with launch-time offsets.
    NCH, NST = 8, 3
    cpts = pts // NCH
    capps = []
    for n in ns:
        app = vk.VkFFTApplication()
        rc = vk.initializeVkFFT(app, vk.VkFFTConfiguration(FFTdim=1, size=[n], numberBatches=cpts // n, device=local_rank,
                                                           normalize=1, userTempBuffer=1, tempBufferSize=cpts * 8,
                                                           specifyOffsetsAtLaunch=1))
        assert rc == 0, (n, vk.getVkFFTErrorString(rc))
        capps.append(app)
    streams = [torch.cuda.Stream(device=dev) for _ in range(NST)]
    ctmps = [tmp[i * cpts:(i + 1) * cpts] for i in range(NST)]

    def e2e_step():
        for c in range(NCH):
            st = streams[c % NST]
            with torch.cuda.stream(st):
                buf[c * cpts:(c + 1) * cpts].copy_(host[c * cpts:(c + 1) * cpts], non_blocking=True)      # pinned host -> HBM
                l = vk.VkFFTLaunchParams(buffer=buf, tempBuffer=ctmps[c % NST], bufferOffset=c * cpts * 8, stream=st.cuda_stream)
                for app in capps:
                    rc = vk.VkFFTAppend(app, -1, l) | vk.VkFFTAppend(app, 1, l)
                    if rc:
                        raise RuntimeError(vk.getVkFFTErrorString(rc))
                host[c * cpts:(c + 1) * cpts].copy_(buf[c * cpts:(c + 1) * cpts], non_blocking=True)      # HBM -> host

    def fork():
        ev = torch.cuda.Event()
        ev.record()
        for st in streams:
            st.wait_event(ev)

    def join():
        for st in streams:
            ev = torch.cuda.Event()
            ev.record(st)
            torch.cuda.current_stream().wait_event(ev)

    fork(); e2e_step(); join()
    barrier()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fork()
    for _ in range(args.e2e_steps):
        e2e_step()
    join()
    b.record()
    barrier()
    ms_e2e = a.elapsed_time(b) / args.e2e_steps
    if dist is not None:
        t = torch.tensor([ms_e2e], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_e2e = float(t.item())
    e2e = {"value": world * fl_step / (ms_e2e * 1e-3) / 1e9, "unit": "GFLOP/s", "h2d_bytes_per_step": nbytes,
           "d2h_bytes_per_step": nbytes, "ms_per_step": ms_e2e, "steps": args.e2e_steps,
           "api": "VkFFTAppend via the C ABI on a pinned host buffer: per step the whole 2 GiB input is copied in and the "
                  "whole result copied out, in 8 batch chunks over 3 streams so copies overlap the 32 transforms"}
    for app in capps:
        vk.deleteVkFFT(app)

    for _, app, _ in apps:
        vk.deleteVkFFT(app)

    # ---- config 5, distributed part: one 2^26-point sequence over all ranks (every rank takes part) ---------------------
    dist_rec = None
    if dist is not None and not args.no_dist:
        del buf, tmp, host
        torch.cuda.empty_cache()
        try:
            dist_rec = bench_dist_2p26(torch, dist, vk, local_rank, rank, world)
        except Exception as e:
            dist_rec = {"error": repr(e)}
        buf = torch.zeros(1, dtype=torch.complex64, device=dev)

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    line = {
        "metric": "batched 1D C2C FP32 throughput (sample_0 sweep N=2^7..2^22, fwd+inv)", "value": value,
        "unit": "GFLOP/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "configs[1]: batched 1D C2C FP32 sweep N=2^7..2^22, batch=2^28/N (2 GiB buffer per GPU), "
                               "in place, forward+inverse per N (reference sample_0 semantics, normalize=1)",
                   "l2": "inputs (2 GiB) larger than L2 (126 MB)", "parallelism": f"batch-sharded x{world}, no collective",
                   "points_per_gpu": pts},
        "roofline": roofline, "e2e": e2e, "gpu_launches": launches_per_step * args.steps * world, "clocks": clocks,
        "kernel_shares": kernel_shares, "per_n": per_n, "roundtrip_rel_err": rt_err, "numa": numa,
    }
    if dist_rec is not None:
        line["dist_2p26"] = dist_rec
    if dumped is not None:
        line["dump_outputs"] = dumped
    if world == 1 and not args.no_cpu:
        line["cpu_baseline"], _ = cpu_baseline()
    else:
        line["cpu_baseline"] = None
    if world == 1 and not args.no_ref_gpu:
        try:
            line["vkfft_cuda_ref"] = vkfft_cuda_reference(torch, buf, ns)
        except Exception as e:
            line["vkfft_cuda_ref"] = {"unavailable": repr(e)}
    if world == 1 and not args.no_configs:
        del buf, tmp, host
        torch.cuda.empty_cache()
        try:
            line["per_config"] = bench_configs(torch, vk, peak, dev)
        except Exception as e:
            line["per_config"] = {"error": repr(e)}
        try:
            line["other_lengths"] = bench_other_lengths(torch, vk, peak, dev)
        except Exception as e:
            line["other_lengths"] = {"error": repr(e)}
    if world == 1 and not args.no_sample0:
        line["sample0"] = sample0_scores(local_rank)
    print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
