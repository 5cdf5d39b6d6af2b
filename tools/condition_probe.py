"""Device time of Corex.impute and score_samples(missing='marginalize') against score_samples at the config-3 shape, at
several missing rates, and of the factor-plus-H build at the config-4 model shape.  Writes one JSON record (default
./condition_probe.json).

  python tools/condition_probe.py [--rows 100000] [--vars 10000] [--factors 100] [--rates 0,0.03,0.3,1] [--reps 5] [--out PATH]

The model is synthetic (tools/score_probe.py's: random moments with Delta > 0); conditioning costs the same whatever the
fitted values are, given the missing pattern.  Inputs are seeded float32 device tensors (4 GB at the default shape, far beyond
the 126 MB L2) whose entries are NaN independently with the given rate.  Times are CUDA events around the call after one
warm-up call, median of --reps; when the warm-up call alone takes longer than --slow-s seconds one timed call follows
instead (the record's "reps" says so).  The per-class row counts of the kernel come from the last call."""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from score_probe import card, synthetic_model  # noqa: E402


def timed(fn, reps, slow_s):
    import torch
    t0 = time.time()
    fn()
    torch.cuda.synchronize()
    if time.time() - t0 > slow_s:
        reps = 1
    ms = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ms.append(a.elapsed_time(b))
    return {"median_ms": float(np.median(ms)), "min_ms": float(np.min(ms)), "max_ms": float(np.max(ms)), "reps": reps}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=100000)
    ap.add_argument("--vars", type=int, default=10000)
    ap.add_argument("--factors", type=int, default=100)
    ap.add_argument("--rates", default="0,0.03,0.3,1")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--slow-s", type=float, default=20.0)
    ap.add_argument("--skip-config4", action="store_true")
    ap.add_argument("--out", default="condition_probe.json")
    a = ap.parse_args()
    import torch
    N, n, m = a.rows, a.vars, a.factors
    rec = {"card": card(), "shape": {"rows": N, "vars": n, "factors": m,
                                     "input": "float32, device-resident, seeded, NaN with probability `rate` per entry"}}
    mdl = synthetic_model(n, m, 0)
    g = torch.Generator(device="cuda").manual_seed(0)
    mean = torch.as_tensor(mdl.theta[0], device="cuda").float()
    sd = torch.as_tensor(mdl.theta[1], device="cuda").float()
    x = torch.randn((N, n), generator=g, device="cuda", dtype=torch.float32) * sd + mean
    rec["score_samples"] = timed(lambda: mdl._scores(x), a.reps, a.slow_s)
    rec["factor_build"] = timed(mdl._lowrank_factor, a.reps, a.slow_s)
    rec["factor_h_build"] = timed(lambda: mdl._lowrank_factor(with_h=True), a.reps, a.slow_s)
    rec["rates"] = {}
    for rate in [float(r) for r in a.rates.split(",")]:
        xr = x.clone()
        if rate > 0:
            xr[torch.rand((N, n), generator=g, device="cuda") < rate] = float("nan")
        r = {"impute": timed(lambda: mdl._conditioned(xr, imputed=True, scores=False), a.reps, a.slow_s)}
        r["marginalize"] = timed(lambda: mdl._conditioned(xr), a.reps, a.slow_s)
        c = mdl._condition_counts
        r["rows_per_class"] = {"nothing_to_solve": int(c[0]), "order_le_64": int(c[1]), "order_le_160": int(c[2]),
                               "order_gt_160": int(c[3]), "path_order_M": int(c[4]), "path_order_m": int(c[5])}
        r["ratio_marginalize_over_score_samples"] = r["marginalize"]["median_ms"] / rec["score_samples"]["median_ms"]
        r["ratio_impute_over_score_samples"] = r["impute"]["median_ms"] / rec["score_samples"]["median_ms"]
        rec["rates"][str(rate)] = r
        print(json.dumps({str(rate): r}), flush=True)
        del xr
        torch.cuda.empty_cache()
    del x
    torch.cuda.empty_cache()
    if not a.skip_config4:
        m4, n4 = 500, 50000
        mdl4 = synthetic_model(n4, m4, 1)
        rec["factor_config4"] = {"shape": {"factors": m4, "vars": n4},
                                 "factor_build": timed(mdl4._lowrank_factor, a.reps, a.slow_s),
                                 "factor_h_build": timed(lambda: mdl4._lowrank_factor(with_h=True), a.reps, a.slow_s)}
    os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(rec, f, indent=1)
    print(json.dumps(rec, indent=1))


if __name__ == "__main__":
    main()
