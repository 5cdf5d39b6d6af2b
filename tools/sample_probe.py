"""Device time of Corex.sample at the config-3 model shape, and of impute(return_std=True) and sample_missing(n_draws=5)
against impute at several missing rates.  Writes one JSON record (default ./sample_probe.json).

  python tools/sample_probe.py [--rows 100000] [--vars 10000] [--factors 100] [--cond-rows 10000] [--rates 0,0.03,0.3,1]
                               [--reps 5] [--out PATH]

The model is tools/score_probe.py's synthetic one (random moments with Delta > 0): sampling and conditioning cost the same
whatever the fitted values are.  sample writes its (rows x vars) float64 output to the device (8 GB at the default shape,
far beyond the 126 MB L2); achieved bytes/s count that one write (the algorithmic minimum; the m x n factor is 8 MB) and
flop/s the 2 rows vars factors of U Z.  A separate torch.profiler pass splits one sample call by kernel.  Conditioning inputs
are seeded float32 device tensors (--cond-rows x vars, 400 MB at the default) whose entries are NaN independently with the
given rate.  Times are CUDA events around the call after one warm-up call, median of --reps."""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from condition_probe import timed  # noqa: E402
from score_probe import card, synthetic_model  # noqa: E402


def kernel_split(fn):
    """CUDA kernel time of one call of fn by kernel name (torch.profiler), in ms."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        if e.device_type.name == "CUDA" and getattr(e, "device_time_total", 0) > 0:
            out[e.key[:90]] = out.get(e.key[:90], 0.0) + e.device_time_total / 1e3
    return dict(sorted(out.items(), key=lambda kv: -kv[1]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=100000)
    ap.add_argument("--vars", type=int, default=10000)
    ap.add_argument("--factors", type=int, default=100)
    ap.add_argument("--cond-rows", type=int, default=10000)
    ap.add_argument("--rates", default="0,0.03,0.3,1")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default="sample_probe.json")
    a = ap.parse_args()
    import torch
    N, n, m = a.rows, a.vars, a.factors
    rec = {"card": card(), "shape": {"rows": N, "vars": n, "factors": m, "cond_rows": a.cond_rows}}
    mdl = synthetic_model(n, m, 0)
    run = lambda: mdl.sample(N, seed=1, return_device=True)
    t = timed(run, a.reps, 1e9)
    nbytes, flops = 8.0 * N * n, 2.0 * N * n * m
    t["bytes_per_s"] = nbytes / (t["median_ms"] / 1e3)
    t["fp64_flop_per_s"] = flops / (t["median_ms"] / 1e3)
    t["algorithmic"] = {"bytes": nbytes, "flops": flops, "what": "one write of rows x vars doubles; U Z (rows x factors x vars)"}
    rec["sample"] = t
    rec["sample_kernels_ms"] = kernel_split(run)
    print(json.dumps({"sample": t, "kernels": rec["sample_kernels_ms"]}), flush=True)
    torch.cuda.empty_cache()
    g = torch.Generator(device="cuda").manual_seed(0)
    mean = torch.as_tensor(mdl.theta[0], device="cuda").float()
    sd = torch.as_tensor(mdl.theta[1], device="cuda").float()
    x = torch.randn((a.cond_rows, n), generator=g, device="cuda", dtype=torch.float32) * sd + mean
    rec["rates"] = {}
    for rate in [float(r) for r in a.rates.split(",")]:
        xr = x.clone()
        if rate > 0:
            xr[torch.rand(tuple(x.shape), generator=g, device="cuda") < rate] = float("nan")
        r = {"impute": timed(lambda: mdl.impute(xr, return_device=True), a.reps, 1e9)}
        r["impute_return_std"] = timed(lambda: mdl.impute(xr, return_std=True, return_device=True), a.reps, 1e9)
        c = mdl._condition_counts
        r["rows_per_class_std"] = {"nothing_to_solve": int(c[0]), "order_le_64": int(c[1]), "order_le_160": int(c[2]),
                                   "order_gt_160": int(c[3]), "path_order_M": int(c[4]), "path_order_m": int(c[5])}
        r["sample_missing_5"] = timed(lambda: mdl.sample_missing(xr, n_draws=5, seed=1, return_device=True), a.reps, 1e9)
        for key in ("impute_return_std", "sample_missing_5"):
            r["ratio_%s_over_impute" % key] = r[key]["median_ms"] / r["impute"]["median_ms"]
        rec["rates"][str(rate)] = r
        print(json.dumps({str(rate): r}), flush=True)
        del xr
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(rec, f, indent=1)
    print(json.dumps(rec, indent=1))


if __name__ == "__main__":
    main()
