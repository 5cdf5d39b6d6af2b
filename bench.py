#!/usr/bin/env python
"""bench.py -- Linear CorEx fit-loop throughput on B200 (the driver's measurement contract).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the reference algorithm on the host cores

A "step" is one fit iteration = one `_update_ns` (reference linearcorex.py:290-334): search direction, one
pass pair over X, backtracking line search, accept.  The workload is BASELINE.json configs[2] -- synthetic
Gaussian latent-factor data, N=100 000 samples x n=10 000 variables, m=100 factors, FP64 mode -- the
configuration the metric is quoted on (configs[0..1] are the reference's CPU-scale parity cases).  With
--gpus N>1 the same N x n problem is row-sharded over the ranks (strong scaling; one all-reduce of the
m*n + m moment partials per pass pair), launched under torchrun, one rank per GPU.

One JSON line on stdout (rank 0).  `value` = fit iterations per second with X~ resident in HBM, timed with
CUDA events around exactly K iterations, max over ranks.  `e2e` = the same metric through the public API
(`Corex(...).fit(x_host)`) with the host->device copy of X, preprocessing, the fit, the final moment export
and the device->host copies all inside the timed region; at config 3 that call runs to the reference's default
stopping rule (tol=1e-5: 410 iterations), i.e. it is exactly `Corex(n_hidden=100).fit(X)` (`--e2e-fit budget` spreads K
iterations over the 7 anneal stages instead).  `roofline` is for the dominant kernel (the two
contractions over X, 93 % of a step: `oz_gemm_kernel`, exact int8 digit-plane products on tcgen05 in the default
FP64-faithful mode `fp64_split`; `dgemm_mma_kernel`, DMMA, with --precision fp64), timed live by CUDA events on the
launching stream.
`target` (default workload only) = the same resident measurement at BASELINE.json's north-star shape, 1M x 20k x 100, rows
sharded over the N ranks, so the driver's scaling record carries that curve too.
`cpu_baseline` / `--impl reference` time one fit iteration of the reference algorithm in float64 on all host cores at the
FULL config-3 size (8 GB of X~): the unmodified reference when $LCX_REFERENCE_ROOT (default /root/reference) exists, else
oracle/corex_oracle.py, its numpy restatement (the GPU box has no /root/reference).  Both legs share one code path.
"""
import argparse
import ctypes as C
import json
import os
import statistics
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (N samples, n variables, m factors)
    "config3": (100000, 10000, 100),     # BASELINE.json configs[2]
    "config4": (1000, 50000, 500),       # configs[3] (gaussianize='outliers')
    "target": (1000000, 20000, 100),     # BASELINE.json target shape; one GPU holds it as 120 GB of int8 digit planes
                                         # (fp64_split / fast, streamed preparation); synthetic rows are drawn on device
    "small": (4000, 2000, 20),
}
METRIC = "fit_iters_per_sec"
UNIT = "it/s"


# ----------------------------------------------------------------------------------------------------
# synthetic data: Gaussian latent-factor model (SURVEY.md 8(d)), row-block seeded so ranks build only
# their own rows
# ----------------------------------------------------------------------------------------------------
def make_rows(n_total, n_vars, n_factors, lo, hi, seed=0, snr=1.0, block=4096, threads=None):
    from concurrent.futures import ThreadPoolExecutor
    out = np.empty((hi - lo, n_vars), dtype=np.float32)
    groups = np.arange(n_vars) % n_factors
    a, b = np.float32(np.sqrt(snr / (1.0 + snr))), np.float32(1.0 / np.sqrt(1.0 + snr))
    first = lo // block

    def fill(bi):
        r0, r1 = max(lo, bi * block), min(hi, (bi + 1) * block)
        rng = np.random.default_rng([seed, bi])
        rows = min(n_total, (bi + 1) * block) - bi * block
        z = rng.standard_normal((rows, n_factors), dtype=np.float32)
        e = rng.standard_normal((rows, n_vars), dtype=np.float32)
        e *= b
        e += a * z[:, groups]
        out[r0 - lo:r1 - lo] = e[r0 - bi * block:r1 - bi * block]

    blocks = list(range(first, (hi + block - 1) // block))
    with ThreadPoolExecutor(max_workers=threads or min(16, os.cpu_count() or 1)) as ex:
        list(ex.map(fill, blocks))
    return out


# ----------------------------------------------------------------------------------------------------
# clocks during the timed region (nvidia-smi fields through NVML)
# ----------------------------------------------------------------------------------------------------
class DeviceRows(object):
    """Row-sliceable synthetic data source drawn on the GPU in fixed blocks (same latent-factor model as make_rows, its own
    counter-based streams): lets the 80 GB float32 target matrix be produced block by block for the streamed preparation."""
    BLOCK = 8192

    def __init__(self, n_total, n_vars, n_factors, lo, hi, seed=0, snr=1.0):
        self.shape = (hi - lo, n_vars)
        self.lo, self.n_factors, self.seed, self.snr = lo, n_factors, seed, snr

    def __getitem__(self, sl):
        import torch
        start, stop = self.lo + sl.start, self.lo + sl.stop
        n_vars = self.shape[1]
        groups = torch.arange(n_vars, device="cuda") % self.n_factors
        a, b = (self.snr / (1.0 + self.snr)) ** 0.5, (1.0 / (1.0 + self.snr)) ** 0.5
        out = torch.empty((stop - start, n_vars), dtype=torch.float32, device="cuda")
        for bi in range(start // self.BLOCK, (stop + self.BLOCK - 1) // self.BLOCK):
            g = torch.Generator(device="cuda")
            g.manual_seed(self.seed * 1000003 + bi)
            z = torch.randn((self.BLOCK, self.n_factors), generator=g, device="cuda", dtype=torch.float32)
            e = torch.randn((self.BLOCK, n_vars), generator=g, device="cuda", dtype=torch.float32)
            e.mul_(b).add_(z[:, groups], alpha=a)
            r0, r1 = max(start, bi * self.BLOCK), min(stop, (bi + 1) * self.BLOCK)
            out[r0 - start:r1 - start] = e[r0 - bi * self.BLOCK:r1 - bi * self.BLOCK]
        return out


_CLOCK_HELPER = r"""
import sys, time
import pynvml
pynvml.nvmlInit()
idx = int(sys.argv[1]); period = float(sys.argv[2])
h = pynvml.nvmlDeviceGetHandleByIndex(idx)
mx = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)
pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
sys.stdout.write("ready %d\n" % mx); sys.stdout.flush()
while True:
    t = time.time()
    try:
        c = pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)
        r = int(pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h))
        sys.stdout.write("%.6f %d %d\n" % (t, c, r)); sys.stdout.flush()
    except Exception:
        pass
    time.sleep(period)
"""


class ClockSampler(object):
    """SM clock and throttle reasons of this rank's GPU, sampled through NVML DURING the timed region -- from a helper
    PROCESS.  An NVML query made inside the benchmarking process takes a driver lock that stalls that process's kernel
    launches for ~0.4 ms, and the queries of the ranks of one box serialise: with in-process sampling the first sample of
    every rank landed at the start of the timed region and cost the 8-GPU run 2-3 ms of its 20 ms window (exchange
    0.23 ms per step over 20 steps against 0.10 over 100).  The helper is started (and NVML initialised) before the timed
    region; its samples are matched to the region by wall-clock time stamps."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
               0x80: "hw_power_brake", 0x2: "applications_clocks_setting", 0x100: "display_clock_setting"}
    PERIOD_S = 0.004

    def __init__(self, index):
        import subprocess
        self.samples, self.mask, self.max_mhz, self.proc, self.t0, self.t1 = [], 0, None, None, None, None
        cvd = os.environ.get("CUDA_VISIBLE_DEVICES", "")
        ids = [v.strip() for v in cvd.split(",") if v.strip()]
        if ids and all(v.isdigit() for v in ids) and index < len(ids):
            index = int(ids[index])  # NVML counts physical devices
        try:
            self.proc = subprocess.Popen([sys.executable, "-c", _CLOCK_HELPER, str(index), str(self.PERIOD_S)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            import select
            ready, _, _ = select.select([self.proc.stdout], [], [], 30.0)  # NVML initialised in the helper (or it died)
            first = self.proc.stdout.readline().split() if ready else []
            if len(first) == 2 and first[0] == "ready":
                self.max_mhz = int(first[1])
            else:
                self._kill()
        except Exception:
            self._kill()

    def _kill(self):
        if self.proc is not None:
            try:
                self.proc.kill()
                self.proc.wait(timeout=5)
            except Exception:
                pass
        self.proc = None

    def __enter__(self):
        self.t0 = time.time()
        return self

    def __exit__(self, *exc):
        self.t1 = time.time()
        if self.proc is None:
            return
        time.sleep(2 * self.PERIOD_S)
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self._kill()
            return
        rows = []
        for line in out.splitlines():
            f = line.split()
            if len(f) == 3:
                try:
                    rows.append((float(f[0]), int(f[1]), int(f[2])))
                except ValueError:
                    pass
        inside = [r for r in rows if self.t0 <= r[0] <= self.t1]
        if not inside and rows:  # a window shorter than one period: the sample closest to it
            mid = 0.5 * (self.t0 + self.t1)
            inside = [min(rows, key=lambda r: abs(r[0] - mid))]
        self.samples = [r[1] for r in inside]
        for r in inside:
            self.mask |= r[2]

    def summary(self):
        return {"sm_mhz": statistics.median(self.samples) if self.samples else None, "sm_max_mhz": self.max_mhz,
                "samples": len(self.samples), "sampler": "NVML in a helper process, every %d ms" % round(self.PERIOD_S * 1e3),
                "reasons": sorted(name for bit, name in self.REASONS.items() if self.mask & bit)}


# ----------------------------------------------------------------------------------------------------
# reference algorithm on the host cores (the only place bench.py executes oracle/)
# ----------------------------------------------------------------------------------------------------
REFERENCE_ROOT = os.environ.get("LCX_REFERENCE_ROOT", "/root/reference")


def host_standardized(n_total, n_vars, n_factors, rows, threads):
    """float64 X~ of the first `rows` synthetic rows: (x - mean) / std per column, built block-wise in threads (the timed
    quantity is the fit iteration; this only has to be quick)."""
    from concurrent.futures import ThreadPoolExecutor
    x32 = make_rows(n_total, n_vars, n_factors, 0, rows, threads=threads)
    blocks = [(lo, min(rows, lo + 2048)) for lo in range(0, rows, 2048)]
    with ThreadPoolExecutor(max_workers=threads) as ex:
        mu = sum(ex.map(lambda b: x32[b[0]:b[1]].sum(axis=0, dtype=np.float64), blocks)) / rows
        sq = sum(ex.map(lambda b: ((x32[b[0]:b[1]] - mu) ** 2).sum(axis=0), blocks))
        sd = np.sqrt(sq / rows).clip(1e-10)
        xt = np.empty((rows, n_vars), dtype=np.float64)

        def fill(b):
            xt[b[0]:b[1]] = (x32[b[0]:b[1]] - mu) / sd
        list(ex.map(fill, blocks))
    return xt


def _reference_stepper(n_factors):
    """(kind, init, step) over the UNMODIFIED reference when LCX_REFERENCE_ROOT exists (its float64 path: the module-global
    numpy shim of oracle/gen_golden.py), else over the oracle port (the GPU box has no /root/reference)."""
    if os.path.isdir(os.path.join(REFERENCE_ROOT, "linearcorex")):
        try:
            sys.path.insert(0, REFERENCE_ROOT)
            import linearcorex.linearcorex as ref

            class _F64(object):
                float32 = np.float64

                def __getattr__(self, name):
                    return getattr(np, name)
            ref.np = _F64()
            mdl = ref.Corex(n_hidden=n_factors, seed=0, tol=1e-12)

            def init(xt, w, eps):
                mdl.n_samples, mdl.nv = xt.shape
                mdl.eps, mdl.ws = eps, w
                mdl.moments = mdl._calculate_moments(xt, w, quick=True)

            def step(xt):
                mdl.ws, mdl.moments = mdl._update_ns(xt)
                return None
            return "reference", init, step, "unmodified %s/linearcorex/linearcorex.py _update_ns (:290-334), float64 path" % REFERENCE_ROOT
        except Exception:
            pass
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import corex_oracle as oc
    state = {}

    def init(xt, w, eps):
        state.update(w=w, eps=eps, m=oc.moments_ns(xt, w, eps))

    def step(xt):
        rec = {}
        state["w"], state["m"] = oc.step_ns(xt, state["w"], state["m"], state["eps"], 1e-12, trace=rec)
        return rec.get("trials")
    return "port", init, step, "oracle/corex_oracle.py step_ns (numpy float64 restatement of linearcorex.py:290-334)"


def time_reference_cpu(n_total, n_vars, n_factors, steps, warmup):
    """Time one fit iteration (`_update_ns`) of the reference algorithm in float64 on the host cores, at the FULL row count
    whenever X~ fits in host memory (config 3: 8 GB), else on the largest row sub-sample that does (cost is linear in N)."""
    try:  # torchrun exports OMP_NUM_THREADS=1 to its workers; the CPU arm must use every host core
        from threadpoolctl import threadpool_limits
        threadpool_limits(limits=os.cpu_count() or 1)
    except Exception:
        pass
    threads = min(32, os.cpu_count() or 1)
    try:
        import psutil
        avail = psutil.virtual_memory().available
    except Exception:
        avail = 64 << 30
    per_row = n_vars * (8 + 4) * 1.6  # float64 X~ + the float32 source + numpy temporaries of a step
    rows = int(min(n_total, max(512, 0.6 * avail / per_row)))
    t0 = time.perf_counter()
    xt = host_standardized(n_total, n_vars, n_factors, rows, threads)
    t_pre = time.perf_counter() - t0
    kind, init, step, what = _reference_stepper(n_factors)
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import corex_oracle as oc
    np.random.seed(0)
    eps = 0.6
    w = np.random.randn(n_factors, n_vars)
    w /= (10. * oc.norm_y(xt, w, 0.0))[:, np.newaxis]
    init(xt, w, eps)
    trials = []
    for _ in range(warmup):
        step(xt)
    t0 = time.perf_counter()
    for _ in range(steps):
        trials.append(step(xt))
    dt = time.perf_counter() - t0
    try:
        from threadpoolctl import threadpool_info
        cores = max([p.get("num_threads", 1) for p in threadpool_info()] + [1])
    except Exception:
        cores = os.cpu_count() or 1
    it_s_sample = steps / dt
    scale = rows / float(n_total)
    tr = [t for t in trials if t is not None]
    return {"value": it_s_sample * scale, "unit": UNIT, "cores": int(cores), "kind": kind,
            "sample": "%s, %d of %d rows x %d vars x %d factors%s, %d iterations after %d warm-up%s; %.4g it/s measured%s; "
                      "building X~ on the host %.1f s (untimed)"
                      % (what, rows, n_total, n_vars, n_factors, " (FULL size)" if rows == n_total else "", steps, warmup,
                         ", %.2f trials/iteration" % float(np.mean(tr)) if tr else "", it_s_sample,
                         "" if rows == n_total else " on the sample, scaled x%.4g (cost linear in N)" % scale, t_pre),
            "ms_per_step_sample": 1e3 * dt / steps, "rows": rows}


def run_reference(args, shape):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n_total, n_vars, n_factors = shape
    # at least 5 warm-up iterations, like the `cpu_baseline` leg of the CUDA arm: the first iterations of a stage backtrack 4-5
    # times (each trial is a full pass pair on the CPU), steady state is 1.3-1.9 trials per iteration
    base = time_reference_cpu(n_total, n_vars, n_factors, args.steps, max(args.warmup, 5))
    line = {"impl": "reference", "metric": METRIC, "value": base["value"], "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 / base["value"], "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_name(args, shape), "n_samples": n_total, "n_variables": n_vars,
                       "n_factors": n_factors, "mode": "numpy float64 on host cores"},
            "cpu_baseline": {k: base[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": base["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


def workload_name(args, shape):
    """The same string in both arms (the driver compares it); the arithmetic of each arm is in config.mode / dtype."""
    return "%s: synthetic latent-factor data N=%d x n=%d, m=%d, FP64 mode" % (args.workload, shape[0], shape[1], shape[2])


MODE_NAMES = {"fp64": "FP64 (DMMA)", "fp64_split": "FP64 (6 int8 radix-254 digit planes on tcgen05)",
              "fp64_split5": "FP64 (5 int8 radix-254 digit planes on tcgen05)",
              "fp64_split7": "FP64 (7 int8 radix-254 digit planes on tcgen05)", "fast": "fast (3 int8 digit planes)"}
DIGITS = {"fp64": 0, "fp64_split": 6, "fp64_split5": 5, "fp64_split7": 7, "fast": 3}


# ----------------------------------------------------------------------------------------------------
# this repo's CUDA path
# ----------------------------------------------------------------------------------------------------
def measure_dgemm_peak(torch):
    n = 6144
    a = torch.randn(n, n, dtype=torch.float64, device="cuda")
    b = torch.randn(n, n, dtype=torch.float64, device="cuda")
    best = 1e30
    for i in range(5):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        torch.matmul(a, b)
        e1.record()
        torch.cuda.synchronize()
        if i > 0:
            best = min(best, e0.elapsed_time(e1))
    return 2.0 * n ** 3 / best / 1e9


def measure_int8_peak(torch, seconds=1.0):
    """int8 tensor throughput measured in this run: cuBLASLt IGEMM 8192^3 (torch._int_mm, int8 x int8 -> int32, random
    operands), best single launch (burst) and back to back for `seconds` (sustained, under the power cap)."""
    try:
        n = 8192
        a = torch.randint(-127, 128, (n, n), dtype=torch.int8, device="cuda")
        b = torch.randint(-127, 128, (n, n), dtype=torch.int8, device="cuda").t()  # column-major B: the TN form
        for _ in range(3):
            torch._int_mm(a, b)
        torch.cuda.synchronize()
        best = 1e30
        for _ in range(5):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            torch._int_mm(a, b)
            e1.record()
            torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1))
        reps = max(8, int(seconds * 1e3 / best))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            torch._int_mm(a, b)
        e1.record()
        torch.cuda.synchronize()
        ops = 2.0 * n ** 3
        return {"burst_tops": ops / best / 1e9, "sustained_tops": ops * reps / e0.elapsed_time(e1) / 1e9,
                "how": "torch._int_mm (cuBLASLt IGEMM) 8192^3, random int8; best of 5 / %d launches back to back" % reps}
    except Exception as exc:  # noqa: BLE001
        return {"burst_tops": None, "sustained_tops": None, "how": "torch._int_mm unavailable: %r" % (exc,)}


def ncu_evidence(precision):
    """Per-launch numbers of the dominant kernel from the newest committed `ncu --set full` summary of this workload
    (profiles/rNN_oz_gemm_ncu_full_config3.csv / rNN_dgemm_ncu_full_config3.csv), identified by file name and hash."""
    import glob
    import hashlib
    pat = "r*_oz_gemm_ncu_full_config3.csv" if precision != "fp64" else "r*_dgemm_ncu_full_config3.csv"
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", pat)))
    if not files:
        return None
    path = files[-1]
    raw = open(path, "rb").read()
    rows = {}
    import csv
    for rec in csv.reader(raw.decode().splitlines()):
        if len(rec) >= 3:
            rows[rec[0]] = rec[1:]
    scale = {"Gbyte": 1e9, "Mbyte": 1e6, "Kbyte": 1e3, "byte": 1.0, "Tbyte": 1e12}

    def vals(name):
        if name not in rows:
            return None
        unit = rows[name][0]
        try:
            return [float(v) * scale.get(unit, 1.0) for v in rows[name][1:]]
        except ValueError:
            return None
    rd, wr = vals("dram__bytes_read.sum"), vals("dram__bytes_write.sum")
    if not rd or not wr:
        return None
    out = {"file": os.path.relpath(path, ROOT), "sha256_16": hashlib.sha256(raw).hexdigest()[:16],
           "kernels": rows.get("metric", ["", ""])[1:],
           "dram_bytes_per_launch": [a + b for a, b in zip(rd, wr)]}
    for key, name in (("delivered_bytes_per_launch", "l1tex__m_xbar2l1tex_read_bytes.sum"),
                      ("tensor_pipe_active_pct", "sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_active"),
                      ("duration_ms_under_ncu", "gpu__time_duration.sum")):
        v = vals(name)
        if v:
            out[key] = v
    return out


DUMP_BYTES = 64 << 20


def dump_outputs(directory, mdl, trace, rank):
    """Write what `Corex.fit` would hand its caller had it stopped after the last timed iteration -- `ws` and every `moments`
    key after the final sort by TC (Corex._finish) -- plus the TC of each timed iteration, as float64 `<name>.npy` files
    (moments keys with punctuation squeezed to `_`).  An array larger than an equal share of DUMP_BYTES is replaced by the
    entries at a fixed, seeded set of flat positions, so two builds run with the same arguments compare element for element."""
    import re
    mdl._finish()  # collective on several ranks: every rank runs it, rank 0 writes
    if rank != 0:
        return
    arrays = {"ws": mdl.ws, "TC_per_step": [t["TC"] for t in trace]}
    for key in list(mdl.moments):
        arrays["moments_" + re.sub(r"[^A-Za-z0-9]+", "_", key).strip("_")] = mdl.moments[key]
    share = DUMP_BYTES // 8 // len(arrays)
    os.makedirs(directory, exist_ok=True)
    for name, value in arrays.items():
        a = np.asarray(value, dtype=np.float64)
        if a.size > share:
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, share, replace=False))]
        np.save(os.path.join(directory, name + ".npy"), a)


def resident_run(torch, dist, shape, args, steps, warmup, world, rank, local, device_source, x_host, lo, hi, algorithm=None,
                 dump_dir=None):
    """Exactly `steps` fit iterations with X~ (or, on the Gram route, X~^T X~ / N) resident in HBM, timed by CUDA events, max
    over ranks.  With `dump_dir` the fitted model is written there afterwards (dump_outputs)."""
    algorithm = algorithm or args.algorithm or "stream"
    from linearcorex_b200 import Corex, _lib
    n_total, n_vars, n_factors = shape

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    x_dev = DeviceRows(n_total, n_vars, n_factors, lo, hi) if device_source else torch.from_numpy(x_host).cuda()
    mdl = Corex(n_hidden=n_factors, seed=0, tol=1e-12, max_iter=10 ** 9, precision=args.precision,
                gaussianize=args.gaussianize, comm=True if world > 1 else None,
                stream_rows=32768 if device_source else None, algorithm=algorithm)
    schedule = mdl._prepare(x_dev)
    prep = dict(mdl.timings)
    del x_dev
    mdl._begin_stage(schedule[0], rescale=False)
    sess = mdl._sess
    def iterate(k):
        """Exactly k iterations of the current stage, the way fit() runs them (lcx_run_stage_ns).  A stage that meets its
        stopping rule (tol = 1e-12) returns early; it is entered again until k iterations have run, so the timed window
        always holds the requested number of steps."""
        n0 = len(mdl.trace)
        while len(mdl.trace) - n0 < k:
            before = len(mdl.trace)
            mdl.max_iter = k - (before - n0)
            if not mdl._run_stage_native() or len(mdl.trace) == before:
                raise RuntimeError("the fit stopped after %d of %d iterations" % (before - n0, k))
        return k

    iterate(warmup)
    sess.lib.lcx_profile_enable(sess.h, 1)
    k1, k2, kx, pairs = C.c_double(), C.c_double(), C.c_double(), C.c_longlong()
    sess.lib.lcx_profile_read_phases(sess.h, C.byref(k1), C.byref(k2), C.byref(kx), C.byref(pairs), 1)
    launches0 = sess.launches()
    n_trace0 = len(mdl.trace)
    clocks = ClockSampler(local)  # helper process up and NVML initialised before the ranks line up
    barrier()
    with clocks:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        iterate(steps)
        e1.record()
        barrier()
    ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = t.item()
    sess.lib.lcx_profile_read_phases(sess.h, C.byref(k1), C.byref(k2), C.byref(kx), C.byref(pairs), 1)
    sess.lib.lcx_profile_enable(sess.h, 0)
    np_ = max(1, pairs.value)
    # every rank must hold bit-identical weights (the replicated line search stays in lock-step only then)
    identical = None
    if world > 1:
        cs = sess.view(_lib.A_W).contiguous().view(torch.int64).sum().reshape(1)
        lo_, hi_ = cs.clone(), cs.clone()
        dist.all_reduce(lo_, op=dist.ReduceOp.MIN)
        dist.all_reduce(hi_, op=dist.ReduceOp.MAX)
        identical = bool((lo_ == hi_).item())
    # per-rank phase times: shows how much of rank 0's `exchange` is waiting for the slowest rank's contractions
    per_rank = None
    if world > 1:
        mine = torch.tensor([k1.value / np_, k2.value / np_, kx.value / np_, e0.elapsed_time(e1) / steps],
                            dtype=torch.float64, device="cuda")
        allr = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(allr, mine)
        per_rank = {"columns": ["k1_ms", "k2_ms", "exchange_ms", "step_ms"],
                    "ranks": [[round(float(v), 4) for v in t.tolist()] for t in allr]}
    trace = mdl.trace[n_trace0:]
    res = {"ms": ms, "per_rank": per_rank, "it_s": steps / (ms / 1e3), "k1_ms": k1.value / np_, "k2_ms": k2.value / np_, "exchange_ms": kx.value / np_,
           "pairs": pairs.value, "launches": sess.launches() - launches0, "prep": prep,
           "trials": float(np.mean([t["trials"] for t in trace])) if trace else 0.0, "tc": float(mdl.tc),
           "clocks": clocks.summary(), "peer": sess._peer_buf is not None, "algorithm": mdl.algorithm_used, "ranks_bit_identical": identical,
           "n_local": hi - lo}
    if dump_dir:
        dump_outputs(dump_dir, mdl, trace, rank)
    del mdl, sess
    torch.cuda.empty_cache()
    return res


def roofline_of(res, shape, args, peaks, dgemm_peak, i8_peak):
    """Roofline record of the two X contractions from the live CUDA-event timings of a resident run."""
    n_total, n_vars, n_factors = shape
    digits = DIGITS[args.precision]
    if os.environ.get("LCX_SPLIT_DIGITS") and digits:
        digits = int(os.environ["LCX_SPLIT_DIGITS"])
    n_local = res["n_local"]
    pair_flops = 4.0 * n_local * n_vars * n_factors           # K1 + K2 of one pass pair on this rank (FP64-equivalent)
    pair_ms = res["k1_ms"] + res["k2_ms"]                      # the two contractions incl. their digit-slicing kernels
    fp64_equiv = pair_flops / (pair_ms / 1e3) / 1e12 if pair_ms > 0 else 0.0
    out = {"bound": "tensor"}
    if digits:
        # split-integer modes: each FP64 multiply-add is S(S+1)/2 exact int8 multiply-adds on tcgen05 (kind::i8)
        pair_ops = pair_flops * digits * (digits + 1) / 2
        achieved = pair_ops / (pair_ms / 1e3) / 1e12 if pair_ms > 0 else 0.0
        peak = 2.0 * float(peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops", 1400.0)))
        out.update(achieved=achieved, peak=peak, unit="TOP/s", frac=achieved / peak,
                   kernel="oz_gemm_kernel<%d,*> (tcgen05.mma kind::i8 + TMA; Y = X~ A^T and X~^T Y as %d int8 digit-plane "
                          "products each, incl. digit slicing of A and Y), %d pass pairs timed by CUDA events"
                          % (digits, digits * (digits + 1) // 2, res["pairs"]),
                   peak_source="2 x bf16_tflops_sustained of MEASURED_PEAKS.json%s (kind::i8 runs at twice the bf16 rate on B200; "
                               "sustained because the kernel is timed inside a long power-capped step; burst would be 2 x %s)"
                               % ("" if "bf16_tflops_sustained" in peaks else " [fallback 1400]", peaks.get("bf16_tflops")))
        if i8_peak and i8_peak.get("sustained_tops"):
            out["int8_peak_measured_in_run"] = i8_peak
            out["frac_of_int8_measured_in_run"] = achieved / i8_peak["sustained_tops"]
        # the kind::i8 pipe alone, operands resident in shared memory, random int8 data (tools/experiments/
        # i8_peak_probe.cu, profiles/r01_i8_peak_probe.txt): 4262 TOP/s burst, 3706 sustained under the power cap
        out["frac_of_measured_i8_pipe_sustained"] = achieved / 3705.6
    else:
        pair_ops = pair_flops
        out.update(achieved=fp64_equiv, peak=dgemm_peak, unit="TFLOP/s", frac=fp64_equiv / dgemm_peak if dgemm_peak else None,
                   kernel="dgemm_mma_kernel (Y = X~ A^T and X~^T Y, DMMA.8x8x4), %d pass pairs timed by CUDA events" % res["pairs"],
                   peak_source="cuBLAS DGEMM 6144^3 measured in this run (MEASURED_PEAKS.json has no FP64 entry; nominal B200 "
                               "FP64 tensor peak is 40 TFLOP/s)")
    out.update(algorithmic_ops_per_pair=pair_ops, fp64_equivalent_tflops=fp64_equiv,
               share_of_step=pair_ms * res["pairs"] / res["ms"] if res["ms"] > 0 else None,
               cublas_dgemm_tflops_in_run=dgemm_peak)
    return out


def gram_record(res, shape, args, peaks, i8_peak, steps):
    """Sub-record of a resident run on the Gram route: the per-iteration product G A^T and the one-off build of G."""
    n_total, n_vars, n_factors = shape
    digits = DIGITS[args.precision]
    planes = digits * (digits + 1) / 2
    gdigits = digits   # the matrix and its operand carry the digits of the data (Corex.GRAM_PRECISION)
    peak = 2.0 * float(peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops", 1400.0)))
    prod_ops = 2.0 * n_vars * n_vars * n_factors * gdigits * (gdigits + 1) / 2   # one n x n x m product as int8 digit-plane products
    prod_ms = res["k1_ms"]
    build_s = res["prep"].get("gram_build_s")
    # the build computes the upper triangle of X~^T X~ on this rank's rows: n (n + block) / 2 outputs, ~half of 2 N n^2
    build_ops = 2.0 * res["n_local"] * n_vars * n_vars * planes / 2.0
    ms_step = res["ms"] / steps
    out = {"what": "Gram route (Corex(algorithm='gram'); 'auto' picks it for N >= n): X~^T X~ / N is formed once from the int8 "
                   "digit planes (exact products on tcgen05, upper triangle), then every pass pair of the fit is ONE "
                   "n x n x m product with it -- results equal to the streaming route and the reference to 1e-9 "
                   "(tests/test_gpu_gram.py)",
           "metric": METRIC, "value": res["it_s"], "unit": UNIT, "ms_per_step": ms_step, "steps": steps,
           "algorithm_used": res.get("algorithm"),
           "phases_ms_per_step": {"product_G_At": res["pairs"] / steps * prod_ms,
                                  "split_k_combine": res["pairs"] / steps * res["exchange_ms"],
                                  "m_x_n_phase_and_host_sync": ms_step - res["pairs"] / steps * (prod_ms + res["k2_ms"] + res["exchange_ms"])},
           "one_off_s": {k: (round(v, 4) if isinstance(v, float) else v) for k, v in res["prep"].items()},
           "roofline_product": {"bound": "tensor", "achieved": prod_ops / (prod_ms / 1e3) / 1e12 if prod_ms > 0 else None,
                                "peak": peak, "unit": "TOP/s",
                                "frac": prod_ops / (prod_ms / 1e3) / 1e12 / peak if prod_ms > 0 else None,
                                "kernel": "oz_gemm_kernel<%d,true,2> (G planes K-major x digit planes of A, %d digits each = %d plane "
                                          "products, output stored factor-major) incl. digit slicing of A"
                                          % (gdigits, gdigits, gdigits * (gdigits + 1) // 2)},
           "trials_per_iteration": res["trials"], "TC_after_timed_region": res["tc"], "clocks": res["clocks"],
           "ranks_bit_identical": res["ranks_bit_identical"], "gpu_launches": int(res["launches"])}
    if build_s:
        out["roofline_build"] = {"bound": "tensor", "achieved": build_ops / build_s / 1e12, "peak": peak, "unit": "TOP/s",
                                 "frac": build_ops / build_s / 1e12 / peak,
                                 "kernel": "oz_gemm_kernel<%d,false,2> over column blocks of X~ (variables on M) + plane transposes, "
                                           "split-K combine, mirror%s" % (digits, "; incl. the sum over ranks" if res["n_local"] < n_total else "")}
        if i8_peak and i8_peak.get("sustained_tops"):
            out["roofline_build"]["frac_of_int8_measured_in_run"] = build_ops / build_s / 1e12 / i8_peak["sustained_tops"]
    return out


def timed_fit(torch, dist, world, kw, x, barrier):
    """One end-to-end `Corex(**kw).fit(x)`: wall seconds (max over ranks) and the fitted model."""
    from linearcorex_b200 import Corex
    barrier()
    mdl = Corex(**kw)
    t0 = time.perf_counter()
    mdl.fit(x)
    torch.cuda.synchronize()
    sec = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([sec], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        sec = t.item()
    return sec, mdl


def run_ours(args, shape):
    import torch
    import torch.distributed as dist
    from linearcorex_b200 import Corex, shard_rows

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    n_total, n_vars, n_factors = shape
    lo, hi = shard_rows(n_total, rank, world)
    device_source = args.workload == "target"   # too large for a host copy in this harness: drawn on the device
    x_host = None if device_source else make_rows(n_total, n_vars, n_factors, lo, hi)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            peaks = json.load(fh)
    except Exception:
        pass
    digits = DIGITS[args.precision]
    dgemm_peak = measure_dgemm_peak(torch) if rank == 0 else 0.0
    i8_peak = measure_int8_peak(torch) if (rank == 0 and digits) else None

    # ---- device-resident timing: exactly K iterations ----------------------------------------------
    res = resident_run(torch, dist, shape, args, args.steps, args.warmup, world, rank, local, device_source, x_host, lo, hi,
                       dump_dir=args.dump_outputs)
    ms, it_s, n_local = res["ms"], res["it_s"], res["n_local"]
    # the Gram route on the same data, as a sub-record (N >= n, split modes): the default of the public API at this shape
    gram = None
    if args.algorithm is None and digits and n_total >= n_vars:
        barrier()
        gres = resident_run(torch, dist, shape, args, args.steps, args.warmup, world, rank, local, device_source, x_host, lo, hi,
                            algorithm="gram")
        gram = gram_record(gres, shape, args, peaks, i8_peak, args.steps)
    exchange = ("none (single rank)" if world == 1 else
                "fused split-K combine + two-shot all-reduce kernel over NVLink peer memory" if res["peer"]
                else "split-K combine kernel + NCCL all-reduce (torch.distributed hook)")

    # ---- end to end through the public API, host buffers in, host results out -----------------------
    per_stage = max(1, args.steps // 7)
    if device_source:
        # the 80 GB target matrix has no host copy in this harness: the public-API run below is fed from the device
        # generator through the streamed preparation (3 passes), so h2d_bytes_per_step is 0 and this is NOT the
        # contract's host-buffer e2e figure -- the default workload (config3) carries that.
        barrier()
        e2e_mdl = Corex(n_hidden=n_factors, seed=0, tol=1e-12, max_iter=per_stage, precision=args.precision,
                        gaussianize=args.gaussianize, comm=True if world > 1 else None, stream_rows=32768,
                        algorithm=args.algorithm or "auto")
        t0 = time.perf_counter()
        e2e_mdl.fit(DeviceRows(n_total, n_vars, n_factors, lo, hi))
        torch.cuda.synchronize()
        e2e_s = time.perf_counter() - t0
        e2e_iters = len(e2e_mdl.history["TC"])
        e2e = {"value": e2e_iters / e2e_s, "unit": UNIT, "h2d_bytes_per_step": 0,
               "d2h_bytes_per_step": int(sum(np.asarray(v).nbytes for v in dict.values(e2e_mdl.moments)) / e2e_iters),
               "iterations": e2e_iters, "seconds": e2e_s, "phases_s": {k: (round(v, 4) if isinstance(v, float) else v) for k, v in e2e_mdl.timings.items()},
               "algorithm": e2e_mdl.algorithm_used,
               "what": "Corex.fit(device row generator), streamed preparation; not a host-buffer e2e (see config3)"}
        del e2e_mdl
        e2e_stream = None
    else:
        # the e2e input lives in page-locked host memory (the contract's "from pinned host memory"); --pageable times
        # the pageable-numpy path (an extra pipelined host memcpy into pinned staging) instead
        x_pin = None if args.pageable else torch.from_numpy(x_host).pin_memory()
        x_in = x_pin if x_pin is not None else x_host
        # "converge" = the call a user makes: Corex(n_hidden=m).fit(X) with the reference's default stopping rule
        # (tol=1e-5, max_iter=10000; 410 iterations at config 3).  "budget" = K iterations spread over the 7 stages.
        converge = args.e2e_fit == "converge"

        def e2e_record(algorithm):
            kw = dict(n_hidden=n_factors, seed=0, precision=args.precision, gaussianize=args.gaussianize,
                      comm=True if world > 1 else None, algorithm=algorithm)
            if not converge:
                kw.update(tol=1e-12, max_iter=per_stage)
            # The timed call is the SECOND fit in this process: one untimed fit of a single iteration per stage runs first,
            # so the caching allocator already holds its blocks (cudaMalloc of ~20 GB costs 0.2-0.3 s the first time) and
            # the NVLink peer mapping exists -- a first call in a fresh process pays ~0.3 s more.
            warm = Corex(**dict(kw, tol=1e-12, max_iter=1))
            warm.fit(x_in)
            del warm
            sec, mdl = timed_fit(torch, dist, world, kw, x_in, barrier)
            iters = len(mdl.history["TC"])
            # large models hand `moments` back with the m x n arrays still on the device (LazyMoments): only what crossed to the
            # host inside the timed region is counted
            pending = mdl.moments.pending() if hasattr(mdl.moments, "pending") else []
            d2h = sum(np.asarray(v).nbytes for v in dict.values(mdl.moments)) + mdl.ws.nbytes + 16 * 8 * 4 * iters
            rec = {"value": iters / sec, "unit": UNIT, "h2d_bytes_per_step": int(x_host.nbytes * world / iters),
                   "d2h_bytes_per_step": int(d2h / iters), "iterations": iters, "seconds": sec,
                   "algorithm": "%s -> %s" % (algorithm, mdl.algorithm_used) if algorithm == "auto" else mdl.algorithm_used,
                   "TC": float(mdl.tc), "phases_s": {k: (round(v, 4) if isinstance(v, float) else v) for k, v in mdl.timings.items()},
                   "moments_keys_left_on_device": pending,
                   "what": "second fit in the process: Corex(n_hidden=%d%s%s).fit(pinned host float32 X): H2D of X, preprocess, "
                           "digit slicing%s, 7 anneal stages%s, final sort + full moments, D2H of ws and every moments key"
                           % (n_factors, "" if converge else ", tol=1e-12, max_iter=%d" % per_stage,
                              "" if algorithm == "auto" else ", algorithm='%s'" % algorithm,
                              ", X~^T X~ / N formed once (Gram route)" if mdl.algorithm_used == "gram" else "",
                              " run to the reference's default stopping rule (tol=1e-5, max_iter=10000)" if converge else "")}
            del mdl
            torch.cuda.empty_cache()
            return rec

        # the headline e2e is the call a user makes (all defaults: algorithm='auto'); when that resolves to the Gram route
        # the same call pinned to the streaming route is timed next to it
        e2e = e2e_record(args.algorithm or "auto")
        e2e_stream = None
        if args.algorithm is None and e2e["algorithm"].endswith("gram"):
            e2e_stream = e2e_record("stream")
        del x_pin
    torch.cuda.empty_cache()

    # ---- the north-star shape (BASELINE.json target: 1M x 20k x 100) as a sub-record of the same line -------------------
    target = None
    custom = bool(args.rows or args.vars or args.factors)
    if args.workload == "config3" and not custom and not args.no_target and digits:
        tshape = WORKLOADS["target"]
        tlo, thi = shard_rows(tshape[0], rank, world)
        tsteps = max(4, min(args.steps, 8))
        barrier()
        tres = resident_run(torch, dist, tshape, args, tsteps, 3, world, rank, local, True, None, tlo, thi)
        trl = roofline_of(tres, tshape, args, peaks, dgemm_peak, i8_peak)
        target = {"workload": "target: synthetic latent-factor data N=%d x n=%d, m=%d, %s mode; rows drawn on the device "
                              "(no 80 GB host copy in this harness), streamed preparation" % (tshape + (MODE_NAMES[args.precision],)),
                  "metric": METRIC, "value": tres["it_s"], "unit": UNIT, "ms_per_step": tres["ms"] / tsteps, "steps": tsteps,
                  "warmup": 3, "n_gpus": world, "rows_per_gpu": tres["n_local"], "scaling": "strong",
                  "updates_per_sec": tres["it_s"] * tshape[0] * tshape[1] * tshape[2],
                  "roofline": {k: trl[k] for k in ("bound", "achieved", "peak", "unit", "frac", "fp64_equivalent_tflops",
                                                   "share_of_step", "frac_of_int8_measured_in_run") if k in trl},
                  "phases_ms": {"k1": tres["k1_ms"], "k2": tres["k2_ms"], "exchange": tres["exchange_ms"],
                                "replicated_and_sync": tres["ms"] / tsteps - tres["pairs"] / tsteps *
                                (tres["k1_ms"] + tres["k2_ms"] + tres["exchange_ms"])},
                  "clocks": tres["clocks"], "TC_after_timed_region": tres["tc"], "prepare_s": {k: (round(v, 3) if isinstance(v, float) else v) for k, v in tres["prep"].items()},
                  "trials_per_iteration": tres["trials"], "ranks_bit_identical": tres["ranks_bit_identical"],
                  "gpu_launches": int(tres["launches"])}
        if args.algorithm is None:
            barrier()
            tg = resident_run(torch, dist, tshape, args, 20, 5, world, rank, local, True, None, tlo, thi, algorithm="gram")
            target["gram"] = gram_record(tg, tshape, args, peaks, i8_peak, 20)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        # same rows, warm-up and code path as `--impl reference` (5 warm-up iterations: the first iterations of a stage
        # backtrack 4-5 times; steady state is 1.3-1.9 trials per iteration), fewer timed steps
        cpu = time_reference_cpu(n_total, n_vars, n_factors, steps=max(4, min(args.steps, 8)), warmup=5)
        cpu = {k: cpu[k] for k in ("value", "unit", "cores", "kind", "sample")}
    rl = roofline_of(res, shape, args, peaks, dgemm_peak, i8_peak)
    k1_ms, k2_ms = res["k1_ms"], res["k2_ms"]
    delivered = None
    if digits:
        # operand tiles landing in shared memory per launch (what ncu reports as l1tex__m_xbar2l1tex_read_bytes): per
        # 128-row M tile and 64-deep K block every factor tile receives the S planes of the X~ tile plus its own factor planes
        bn = 128 if digits <= 4 else 64
        per_block = digits * 64 * (128 * -(-n_factors // bn) + 16 * -(-n_factors // 16))
        b1 = -(-n_local // 128) * -(-n_vars // 64) * per_block
        b2 = -(-n_vars // 128) * -(-n_local // 64) * per_block
        delivered = {"bytes_per_launch_model": [b1, b2],
                     "tb_per_s": [b1 / (k1_ms * 1e9) if k1_ms > 0 else None, b2 / (k2_ms * 1e9) if k2_ms > 0 else None]}
    # evidence from the committed ncu capture of this exact workload (config 3, one GPU): DRAM traffic per launch and what
    # limits the kernel -- read from the file, never typed in
    ev = ncu_evidence(args.precision) if (args.workload == "config3" and not custom and world == 1) else None
    algo_bytes = n_local * n_vars * (digits if digits else 8)
    traffic = args.traffic
    limiter = None
    if ev is not None:
        if traffic is None:
            traffic = float(np.mean(ev["dram_bytes_per_launch"]))
        limiter = "%s (sha256 %s): DRAM %s GB per launch vs %.2f GB algorithmic" % (
            ev["file"], ev["sha256_16"], "/".join("%.2f" % (v / 1e9) for v in ev["dram_bytes_per_launch"]), algo_bytes / 1e9)
        if "tensor_pipe_active_pct" in ev:
            limiter += "; tensor pipe %s %% of active cycles" % "/".join("%.1f" % v for v in ev["tensor_pipe_active_pct"])
        if "delivered_bytes_per_launch" in ev:
            limiter += "; operand delivery L2->SM %s GB per launch (%.2fx the algorithmic operand bytes)" % (
                "/".join("%.2f" % (v / 1e9) for v in ev["delivered_bytes_per_launch"]),
                float(np.mean(ev["delivered_bytes_per_launch"])) / algo_bytes)
    rl.update(traffic=traffic, limiter=limiter, ncu_evidence=ev, operand_delivery=delivered,
              kernel=rl["kernel"] + "; K1 %.3f ms, K2 %.3f ms per launch" % (k1_ms, k2_ms))
    pair_total = res["pairs"] / args.steps * (k1_ms + k2_ms + res["exchange_ms"])
    line = {
        "metric": METRIC, "value": it_s, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": {"fp64": "f64", "fp64_split": "f64 (6 int8 digit planes = 48 bits, exact int32 products, f64 recombination)",
                  "fp64_split5": "f64 (5 int8 digit planes = 40 bits, exact int32 products, f64 recombination)",
                  "fp64_split7": "f64 (7 int8 digit planes = 56 bits, exact int32 products, f64 recombination)",
                  "fast": "3 int8 digit planes = 24 bits (fp32-equivalent), f64 elsewhere"}[args.precision], "data": "synthetic",
        "config": {"workload": workload_name(args, shape), "mode": MODE_NAMES[args.precision], "n_samples": n_total,
                   "n_variables": n_vars, "n_factors": n_factors, "rows_per_gpu": n_local,
                   "parallelism": "sample-sharded x%d" % world, "exchange_per_pass_pair": exchange,
                   "l2": "inputs_exceed_l2 (X~ block is %.1f GB per GPU)"
                         % (n_local * n_vars * (8 if args.precision == "fp64" else digits) / 1e9),
                   "prepare_s": {k: (round(v, 3) if isinstance(v, float) else v) for k, v in res["prep"].items()},
                   "trials_per_iteration": res["trials"], "TC_after_timed_region": res["tc"]},
        "updates_per_sec": it_s * n_total * n_vars * n_factors,
        "phases_ms_per_step": {"k1": res["pairs"] / args.steps * k1_ms, "k2": res["pairs"] / args.steps * k2_ms,
                               "exchange_incl_split_k_combine": res["pairs"] / args.steps * res["exchange_ms"],
                               "replicated_mxn_phase_and_host_sync": ms / args.steps - pair_total},
        "ranks_bit_identical": res["ranks_bit_identical"],
        "phases_ms_per_rank": res.get("per_rank"),
        "roofline": rl,
        "clocks": res["clocks"],
        "e2e": e2e,
        "gpu_launches": int(res["launches"]),
    }
    if res.get("algorithm") == "gram":  # --algorithm gram: the main arm itself ran the Gram route
        g = gram_record(res, shape, args, peaks, i8_peak, args.steps)
        line["roofline"] = dict(g["roofline_product"], share_of_step=g["phases_ms_per_step"]["product_G_At"] / g["ms_per_step"],
                                build=g.get("roofline_build"), traffic=None)
        line["phases_ms_per_step"] = g["phases_ms_per_step"]
        line["config"]["algorithm"] = "gram"
    else:
        line["config"]["algorithm"] = "stream (every pass pair reads X~: the north star's formulation); see `gram` for the route "\
                                      "the public API picks at this shape"
    if gram is not None:
        line["gram"] = gram
    if e2e_stream is not None:
        line["e2e_stream"] = e2e_stream
    if target is not None:
        line["target"] = target
    if cpu is not None:
        line["cpu_baseline"] = cpu
    emit(line)
    if world > 1:
        dist.destroy_process_group()


_REAL_STDOUT = None


def emit(line):
    """The one JSON line, on the real stdout (fd 1 is pointed at stderr while the run is in progress so that native
    libraries -- NCCL prints its version banner to stdout -- cannot pollute the contract line)."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=42)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="config3", choices=sorted(WORKLOADS))
    ap.add_argument("--precision", default="fp64_split", choices=["fp64", "fp64_split", "fp64_split5", "fp64_split7", "fast"])
    ap.add_argument("--gaussianize", default="standard")
    ap.add_argument("--algorithm", default=None, choices=["stream", "gram", "auto"],
                    help="stream: every pass pair reads X~ (the north star's formulation); gram: X~^T X~ / N formed once.  "
                         "Default: `value` / `roofline` / `target` time the streaming route, `gram` sub-records time the Gram "
                         "route, and `e2e` is the all-defaults public call (algorithm='auto')")
    ap.add_argument("--rows", type=int, default=0)
    ap.add_argument("--vars", type=int, default=0)
    ap.add_argument("--factors", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-target", action="store_true", help="skip the 1M x 20k x 100 sub-record of the default workload")
    ap.add_argument("--pageable", action="store_true", help="e2e input as a pageable numpy array instead of pinned memory")
    ap.add_argument("--e2e-fit", default=None, choices=["converge", "budget"],
                    help="end-to-end fit: run to the default stopping rule (default for config3) or K iterations over the stages")
    ap.add_argument("--traffic", type=float, default=None, help="dram bytes per launch from an ncu capture, if known")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed iterations, write the fitted ws and moments of that run to DIR/<name>.npy (float64, "
                         "at most 64 MB; larger arrays as a fixed, seeded sample of their entries)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(3, args.warmup)
    shape = list(WORKLOADS[args.workload])
    for i, v in enumerate((args.rows, args.vars, args.factors)):
        if v:
            shape[i] = v
    if args.workload == "config4":
        args.gaussianize = "outliers"
    if args.e2e_fit is None:
        args.e2e_fit = "converge" if args.workload == "config3" and not (args.rows or args.vars or args.factors) else "budget"
    if args.impl == "reference":
        run_reference(args, tuple(shape))
    else:
        run_ours(args, tuple(shape))


if __name__ == "__main__":
    main()
