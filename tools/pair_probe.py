"""Device time of the two X contractions (K1: Y = X~ A^T, K2: X~^T Y) for one shape and mode, from the library's own CUDA
events (lcx_profile_read_phases), on random data drawn on the device.  The library reads the experiment knob LCX_OZ_DEBUG
from the environment (it switches the MMAs / the loads off).

    python tools/pair_probe.py [N n m [precision [repeats]]]        # one JSON line
"""
import ctypes as C
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from linearcorex_b200 import _lib  # noqa: E402
from linearcorex_b200.corex import _DeviceSession  # noqa: E402


def main():
    a = sys.argv[1:]
    N, n, m = (int(v) for v in (a[:3] if len(a) >= 3 else (100000, 10000, 100)))
    prec = a[3] if len(a) >= 4 else "fp64_split"
    reps = int(a[4]) if len(a) >= 5 else 10
    sess = _DeviceSession(_lib.PRECISIONS[prec])
    lib = sess.lib
    ld = lib.lcx_ld(n)
    g = torch.Generator(device="cuda")
    g.manual_seed(0)
    xt = torch.zeros(N, ld, dtype=torch.float64, device="cuda")
    rows = max(1, (1 << 28) // ld)
    for lo in range(0, N, rows):
        hi = min(N, lo + rows)
        xt[lo:hi, :n] = torch.randn(hi - lo, n, generator=g, device="cuda", dtype=torch.float64)
    sess.bind(xt, N, n, m, None)
    del xt
    torch.cuda.empty_cache()
    w = sess.view(_lib.A_W)
    w.copy_(torch.randn(m, n, generator=g, device="cuda", dtype=torch.float64) / (10 * n ** 0.5))
    out_arr = sess.view(_lib.A_GRAD)
    for _ in range(3):
        _lib.check(lib.lcx_sig(sess.h, w.data_ptr(), 0.0, out_arr.data_ptr()))
    torch.cuda.synchronize()
    lib.lcx_profile_enable(sess.h, 1)
    k1, k2, kx, pairs = C.c_double(), C.c_double(), C.c_double(), C.c_longlong()
    lib.lcx_profile_read_phases(sess.h, C.byref(k1), C.byref(k2), C.byref(kx), C.byref(pairs), 1)
    # SM clock and board power while the pairs run (NVML, sampled every 20 ms from a thread): tells a kernel held back by the
    # power cap (clock far below the 1965 MHz maximum at ~1 kW) from one that stalls at full clock
    import threading
    import time
    samples, stop = [], threading.Event()
    try:
        import pynvml
        pynvml.nvmlInit()
        hnd = pynvml.nvmlDeviceGetHandleByIndex(torch.cuda.current_device())

        def poll():
            while not stop.is_set():
                samples.append((pynvml.nvmlDeviceGetClockInfo(hnd, pynvml.NVML_CLOCK_SM), pynvml.nvmlDeviceGetPowerUsage(hnd) / 1e3))
                time.sleep(0.02)
        th = threading.Thread(target=poll, daemon=True)
        th.start()
    except Exception:
        th = None
    for _ in range(reps):
        _lib.check(lib.lcx_sig(sess.h, w.data_ptr(), 0.0, out_arr.data_ptr()))
    lib.lcx_profile_read_phases(sess.h, C.byref(k1), C.byref(k2), C.byref(kx), C.byref(pairs), 1)
    stop.set()
    if th is not None:
        th.join()
    p = max(1, pairs.value)
    knobs = {k: v for k, v in os.environ.items() if k.startswith("LCX_")}
    print(json.dumps({"shape": [N, n, m], "precision": prec, "knobs": knobs, "k1_ms": round(k1.value / p, 4),
                      "k2_ms": round(k2.value / p, 4), "combine_ms": round(kx.value / p, 4), "pairs": p,
                      "sm_mhz_median": sorted(c for c, _ in samples[len(samples) // 3:])[len(samples[len(samples) // 3:]) // 2] if samples else None,
                      "power_w_median": sorted(w_ for _, w_ in samples[len(samples) // 3:])[len(samples[len(samples) // 3:]) // 2] if samples else None,
                      "nvml_samples": len(samples)}))


if __name__ == "__main__":
    main()
