"""Cost of per-row sample weights in Corex.fit at the config-3 shape, on both routes, and of Bayesian-bootstrap refits.
Writes one JSON record (default ./weighted_probe.json).

  python tools/weighted_probe.py [--rows 100000] [--vars 10000] [--factors 100] [--max-iter 40] [--reps 2] [--boot 10]
                                 [--out PATH]

Input: seeded latent-factor data generated on the device as float32 (4 GB at the default shape, far beyond the 126 MB L2),
so every fit reads the same resident tensor.  For each route ('stream', 'gram'; precision fp64_split) the probe fits without
weights, with seeded uniform(0.5, 1.5) weights, and with all-ones weights, alternating the first two --reps times; each fit
runs --max-iter iterations per annealing stage at most (the loop is the same code with and without weights, so a capped fit
measures its rate as well as a converged one).  A fit's wall time ends in a device synchronise; `timings` are the model's
own (preprocess_s, bind_s, gram_build_s, finish_s), and the loop's rate is iterations over the rest of the wall time.  The
all-ones fit is compared bit for bit with the unweighted one.  Then --boot Bayesian-bootstrap refits (weights N times a
flat Dirichlet draw) of the same tensor on the route 'auto' picks, with the stability of clusters() against the full fit."""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from score_probe import card  # noqa: E402


def device_data(N, n, k, seed):
    """X[:, i] = (sqrt(s) Z[:, i mod k] + noise) / sqrt(1 + s), s = 1 + 0.4 (i mod k): the survey's generator, on the device."""
    import torch
    g = torch.Generator(device="cuda").manual_seed(seed)
    z = torch.randn((N, k), generator=g, device="cuda", dtype=torch.float32)
    grp = torch.arange(n, device="cuda") % k
    s = 1.0 + 0.4 * grp.float()
    x = torch.randn((N, n), generator=g, device="cuda", dtype=torch.float32)
    x.add_(z[:, grp] * s.sqrt()).div_((1.0 + s).sqrt())
    return x


def fit(x, w, **kw):
    import torch
    from linearcorex_b200 import Corex
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    mdl = Corex(**kw).fit(x, sample_weight=w)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    t = {k: round(float(v), 5) for k, v in mdl.timings.items() if k in ("upload_s", "preprocess_s", "bind_s", "gram_build_s",
                                                                        "gram_bind_s", "finish_s")}
    it = len(mdl.history.get("TC", []))
    loop = wall - sum(t.values())
    return mdl, {"wall_s": round(wall, 4), "timings": t, "iterations": it, "loop_s": round(loop, 4),
                 "iterations_per_s": round(it / loop, 2) if loop > 0 else None, "algorithm_used": mdl.algorithm_used}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=100000)
    ap.add_argument("--vars", type=int, default=10000)
    ap.add_argument("--factors", type=int, default=100)
    ap.add_argument("--max-iter", type=int, default=40)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--boot", type=int, default=10)
    ap.add_argument("--out", default="weighted_probe.json")
    a = ap.parse_args()
    import torch
    N, n, m = a.rows, a.vars, a.factors
    rec = {"card": card(), "shape": {"rows": N, "vars": n, "factors": m, "max_iter_per_stage": a.max_iter,
                                     "input": "float32, device-resident, seeded latent-factor data (k = 20)"}}
    x = device_data(N, n, 20, 0)
    w = np.random.RandomState(1).uniform(0.5, 1.5, size=N)
    base = dict(n_hidden=m, seed=0, max_iter=a.max_iter, precision="fp64_split", input_dtype="float32")
    fit(device_data(4096, 512, 8, 1), None, **dict(base, n_hidden=8, algorithm="stream"))  # warm-up: module load, first launches
    fit(device_data(4096, 512, 8, 1), w[:4096], **dict(base, n_hidden=8, algorithm="gram"))
    rec["routes"] = {}
    for algorithm in ("stream", "gram"):
        kw = dict(base, algorithm=algorithm)
        r = {"unweighted": [], "weighted": []}
        for _ in range(a.reps):
            r["unweighted"].append(fit(x, None, **kw)[1])
            r["weighted"].append(fit(x, w, **kw)[1])
        plain, _ = fit(x, None, **kw)
        ones, _ = fit(x, np.ones(N), **kw)
        r["all_ones_bit_identical"] = bool(np.array_equal(plain.ws, ones.ws) and
                                           list(plain.history["TC"]) == list(ones.history["TC"]))
        rec["routes"][algorithm] = r
        print(algorithm, json.dumps(r), flush=True)
    kw = dict(base, max_iter=2000)
    full, rec["bootstrap_full_fit"] = fit(x, None, **kw)
    rng = np.random.RandomState(2)
    boots, agree = [], []
    t0 = time.perf_counter()
    for _ in range(a.boot):
        bw = rng.standard_exponential(N)
        bw *= N / bw.sum()
        mdl, info = fit(x, bw, **kw)
        boots.append(info)
        agree.append(float(np.mean(mdl.clusters() == full.clusters())))
    rec["bootstrap"] = {"refits": a.boot, "total_s": round(time.perf_counter() - t0, 3), "fits": boots,
                        "clusters_agreement_with_full_fit": agree,
                        "note": "clusters() labels are factor indices sorted by TCs; agreement is label-for-label"}
    out = a.out
    os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
    with open(out, "w") as f:
        json.dump(rec, f, indent=1)
    print(json.dumps({k: v for k, v in rec.items() if k != "routes"})[:2000])


if __name__ == "__main__":
    main()
