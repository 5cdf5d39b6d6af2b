"""Device time of Corex.conditional (ConditionalGaussian) at the config-3 shape for several target-set sizes |T|, against
Corex.score_samples on full rows and Corex.impute of the same rows with T set to NaN, and of the pattern build at the config-4
model shape.  Writes one JSON record (default ./conditional_probe.json).

  python tools/conditional_probe.py [--rows 100000] [--vars 10000] [--factors 100] [--targets 1,300,3000,9900] [--reps 5]
                                    [--out PATH]

The model is synthetic (tools/score_probe.py's: random moments with Delta > 0); conditioning costs the same whatever the fitted
values are.  T is a seeded random column set and O its complement.  Inputs are seeded float32 device tensors (x_O is up to 4 GB,
far beyond the 126 MB L2).  Times are CUDA events around the call after one warm-up call, median of --reps; impute, which takes
seconds, runs once after its warm-up (the record's "reps" says so)."""
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


def split(n, nt, seed):
    perm = np.random.RandomState(seed).permutation(n)
    return np.sort(perm[nt:]), perm[:nt]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=100000)
    ap.add_argument("--vars", type=int, default=10000)
    ap.add_argument("--factors", type=int, default=100)
    ap.add_argument("--targets", default="1,300,3000,9900")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--skip-config4", action="store_true")
    ap.add_argument("--out", default="conditional_probe.json")
    a = ap.parse_args()
    import torch
    N, n, m = a.rows, a.vars, a.factors
    rec = {"card": card(), "shape": {"rows": N, "vars": n, "factors": m,
                                     "input": "float32, device-resident, seeded; x_O = the observed columns, contiguous"}}
    mdl = synthetic_model(n, m, 0)
    g = torch.Generator(device="cuda").manual_seed(0)
    mean = torch.as_tensor(mdl.theta[0], device="cuda").float()
    sd = torch.as_tensor(mdl.theta[1], device="cuda").float()
    x = torch.randn((N, n), generator=g, device="cuda", dtype=torch.float32) * sd + mean
    rec["corex_score_samples_full_rows"] = timed(lambda: mdl._scores(x), a.reps, 1e9)
    rec["targets"] = {}
    for nt in [int(t) for t in a.targets.split(",")]:
        obs, tgt = split(n, nt, nt)
        xo = x[:, torch.as_tensor(obs, device="cuda")].contiguous()
        cg = mdl.conditional(obs, tgt)
        r = {"n_obs": len(obs), "n_targets": nt,
             "build": timed(lambda: mdl.conditional(obs, tgt), a.reps, 1e9),
             "predict": timed(lambda: cg.predict(xo, return_device=True), a.reps, 1e9),
             "score_samples": timed(lambda: cg._conditioned(xo, False, True), a.reps, 1e9),
             "sample_1_draw": timed(lambda: cg.sample(xo, n_draws=1, seed=1, return_device=True), a.reps, 1e9),
             "flops_per_row_predict": 2.0 * m * (len(obs) + nt),
             "bytes_predict": {"read_x_obs": N * len(obs) * 4, "write_pred": N * nt * 8}}
        del xo
        holes = x.clone()
        holes[:, torch.as_tensor(tgt, device="cuda")] = float("nan")
        r["corex_impute_same_rows"] = timed(lambda: mdl._conditioned(holes, imputed=True, scores=False), 1, 0.0)
        c = mdl._condition_counts
        r["impute_rows_per_class"] = {"order_le_64": int(c[1]), "order_le_160": int(c[2]), "order_gt_160": int(c[3]),
                                      "path_order_M": int(c[4]), "path_order_m": int(c[5])}
        r["ratio_predict_over_score_samples_full"] = r["predict"]["median_ms"] / rec["corex_score_samples_full_rows"]["median_ms"]
        r["ratio_impute_over_predict"] = r["corex_impute_same_rows"]["median_ms"] / r["predict"]["median_ms"]
        rec["targets"][str(nt)] = r
        print(json.dumps({str(nt): r}), flush=True)
        del holes, cg
        torch.cuda.empty_cache()
    del x
    torch.cuda.empty_cache()
    if not a.skip_config4:
        m4, n4 = 500, 50000
        mdl4 = synthetic_model(n4, m4, 1)
        rec["build_config4"] = {}
        for nt in (300, 1500):
            obs, tgt = split(n4, nt, nt)
            rec["build_config4"][str(nt)] = {"shape": {"factors": m4, "vars": n4, "n_obs": len(obs), "n_targets": nt},
                                             "build": timed(lambda: mdl4.conditional(obs, tgt), a.reps, 1e9),
                                             "flops": 2.0 * m4 * m4 * len(obs) + 1.0 * m4 * m4 * n4 + m4 ** 3 / 3.0}
        rec["build_config4"]["corex_factor_build"] = timed(mdl4._lowrank_factor, a.reps, 1e9)
    os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(rec, f, indent=1)
    print(json.dumps(rec, indent=1))


if __name__ == "__main__":
    main()
