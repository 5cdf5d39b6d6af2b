"""Device time of Corex.score_samples against transform and against the dense route, at the config-3 shape, and of the factor
build at the config-4 model shape.  Writes one JSON record (default ./score_probe.json).

  python tools/score_probe.py [--rows 100000] [--vars 10000] [--factors 100] [--reps 5] [--out PATH]

The models are synthetic (random moments with Delta > 0, random ws): scoring and transform cost the same whatever the fitted
values are.  Inputs are seeded float32 device tensors (4 GB at the default shape, far beyond the 126 MB L2).  Times are CUDA
events around the call after one warm-up call, median of --reps; bytes and flops are computed from the shapes."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    import torch
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        info["nvidia_smi"] = q
    except Exception as exc:  # noqa: BLE001 -- the record says what could not be read
        info["nvidia_smi"] = "unavailable: %r" % (exc,)
    return info


def timed(fn, reps):
    import torch
    fn()
    torch.cuda.synchronize()
    ms = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ms.append(a.elapsed_time(b))
    return {"median_ms": float(np.median(ms)), "min_ms": float(np.min(ms)), "max_ms": float(np.max(ms)), "reps": reps}


def synthetic_model(n, m, seed):
    from linearcorex_b200 import Corex
    rng = np.random.RandomState(seed)
    z = rng.randn(m, n)
    z *= np.sqrt(0.8 * rng.uniform(0.2, 1.0, n)) / np.linalg.norm(z, axis=0)
    si = rng.rand(n)
    mdl = Corex(n_hidden=m, precision="fp64")
    mdl.nv, mdl.eps = n, 0.0
    mdl.theta = (rng.randn(n), 0.5 + rng.rand(n))
    mdl.moments = {"rhoinvrho": z * (1 + si), "Si": si}
    mdl.ws = rng.randn(m, n) / np.sqrt(n)
    return mdl


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=100000)
    ap.add_argument("--vars", type=int, default=10000)
    ap.add_argument("--factors", type=int, default=100)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default="score_probe.json")
    a = ap.parse_args()
    import torch
    N, n, m = a.rows, a.vars, a.factors
    rec = {"card": card(), "shape": {"rows": N, "vars": n, "factors": m, "input": "float32, device-resident, seeded"}}
    mdl = synthetic_model(n, m, 0)
    g = torch.Generator(device="cuda").manual_seed(0)
    mean = torch.as_tensor(mdl.theta[0], device="cuda").float()
    sd = torch.as_tensor(mdl.theta[1], device="cuda").float()
    x = torch.randn((N, n), generator=g, device="cuda", dtype=torch.float32) * sd + mean
    ld = ((n + 15) // 16) * 16
    rec["score_samples"] = {
        "factor_build": timed(mdl._lowrank_factor, a.reps),
        "scores_total_device": timed(lambda: mdl._scores(x), a.reps),
        "score_samples_public": timed(lambda: mdl.score_samples(x), a.reps),
        "bytes_per_call": {"read_x": N * n * 4, "write_xt": N * ld * 8, "read_xt": N * ld * 8},
        "flops_projection": 2.0 * N * n * m,
        "flops_factor": 2.0 * m * m * n + 1.0 * m * m * n + m ** 3 / 3.0,
    }
    s = rec["score_samples"]
    s["per_block_ms"] = s["scores_total_device"]["median_ms"] - s["factor_build"]["median_ms"]
    s["per_block_GB_per_s"] = sum(s["bytes_per_call"].values()) / (s["per_block_ms"] * 1e-3) / 1e9
    rec["transform"] = timed(lambda: mdl.transform(x, return_device=True), a.reps)
    rec["ratio_score_over_transform"] = s["scores_total_device"]["median_ms"] / rec["transform"]["median_ms"]

    # the dense route at the same n: materialise Sigma, Cholesky, one triangular solve over the centred rows
    cov = torch.empty((n, n), dtype=torch.float64, device="cuda")
    xc = ((x.double() - torch.as_tensor(mdl.theta[0], device="cuda"))).t().contiguous()
    state = {}

    def dense_cov():
        mdl.get_covariance(out=cov)

    def dense_chol():
        state["L"] = torch.linalg.cholesky(cov)

    def dense_solve():
        torch.linalg.solve_triangular(state["L"], xc, upper=False)
    rec["dense"] = {"get_covariance_ms": timed(dense_cov, a.reps), "cholesky_ms": timed(dense_chol, a.reps),
                    "solve_triangular_ms": timed(dense_solve, a.reps), "flops_cholesky": n ** 3 / 3.0,
                    "flops_solve": 1.0 * n * n * N, "note": "torch.linalg (vendor library) for comparison only"}
    rec["dense"]["total_ms"] = sum(rec["dense"][k]["median_ms"] for k in ("get_covariance_ms", "cholesky_ms", "solve_triangular_ms"))
    del cov, xc, state, x
    torch.cuda.empty_cache()

    m4, n4 = 500, 50000
    mdl4 = synthetic_model(n4, m4, 1)
    rec["factor_config4"] = {"shape": {"factors": m4, "vars": n4}, "factor_build": timed(mdl4._lowrank_factor, a.reps),
                             "flops": 2.0 * m4 * m4 * n4 + 1.0 * m4 * m4 * n4 + m4 ** 3 / 3.0}
    os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(rec, f, indent=1)
    print(json.dumps(rec, indent=1))


if __name__ == "__main__":
    main()
