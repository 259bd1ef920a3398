"""Time of predict(method="lowrank") against the dense conditional predict (DESIGN.md 4.6).

    python scripts/bench_predict_lowrank.py [--out FILE] [--reps N]

Writes one JSON file with the card name and power limit.  The routes are timed alternately in the same
process with CUDA events around whole calls (Ylm moments included: a new process object per call) and
per-stage CUDA events (StarryProcess._stage_ms).  Workloads, B = 64 hyperparameter draws (bench.py, seed 7),
one light curve, conditional branch, limb-darkened, predicted at nts = nt points spread over the data and
beyond it:
  nt1000, nt4096   dense (full covariance), rank 31 with the full covariance, rank 31 with the variance only
  nt1e5            rank 31 with the variance only (one dense K would take 80 GB)
"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
import bench  # noqa: E402
import starry_process_b200 as spb  # noqa: E402
from bench_lowrank import card, timed  # noqa: E402

U_LD = [0.4, 0.26]
ROUTES = {"dense": dict(method="dense", return_cov="full"),
          "lowrank_full": dict(method="lowrank", return_cov="full"),
          "lowrank_diag": dict(method="lowrank", return_cov="diag")}


def workload(name, nt, routes, reps, hp, dev):
    rng = np.random.default_rng(nt)
    t = torch.tensor(np.sort(rng.uniform(0.0, 30.0, nt)), device=dev)
    ts = torch.tensor(np.linspace(-1.0, 31.0, nt), device=dev)
    f = torch.tensor(1e-3 * rng.standard_normal(nt), device=dev)

    def call(route, stage):
        gp = spb.StarryProcess(marginalize_over_inclination=False, normalized=False, **hp)
        gp._stage_ms = stage
        return gp.predict(t, f, 1e-6, t_sample=ts, i=60.0, p=1.0, u=U_LD, **ROUTES[route])

    res = {"B": len(hp["r"]), "nt": nt, "nts": nt}
    out, times, stages = {}, {r: [] for r in routes}, {r: {} for r in routes}
    torch.cuda.reset_peak_memory_stats()
    for k in range(reps + 1):   # call 0 of every route is the warm-up
        for r in routes:
            ms, st, o = timed(lambda stage, r=r: call(r, stage))
            out[r] = o
            if k > 0:
                times[r].append(ms)
                for s, v in st.items():
                    stages[r].setdefault(s, []).append(v)
    for r in routes:
        res[r] = {"ms": times[r], "median_ms": float(np.median(times[r])),
                  "stage_median_ms": {s: float(np.median(v)) for s, v in stages[r].items()}}
    res["peak_allocated_GB"] = torch.cuda.max_memory_allocated() / 1e9
    res["all_finite"] = all(bool(torch.isfinite(x).all()) for o in out.values() for x in o)
    if "dense" in routes:
        mu_d, K_d = (x.cpu().numpy() for x in out["dense"])
        mu_l, K_l = (x.cpu().numpy() for x in out["lowrank_full"])
        scale = np.abs(np.diagonal(K_d, axis1=1, axis2=2)).max()
        res["max_rel_diff_mean"] = float(np.abs(mu_l - mu_d).max() / np.abs(mu_d).max())
        res["max_diff_cov_over_max_var"] = float(np.abs(K_l - K_d).max() / scale)
    print(name, json.dumps(res), flush=True)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="bench_predict_lowrank.json",
                    help="JSON result file (default: ./bench_predict_lowrank.json)")
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_predict_lowrank.py measures on a CUDA device; none is available")
    dev = torch.device("cuda", 0)
    hp = {k: torch.tensor(v[:64], device=dev) for k, v in bench.synthetic_inputs(4096, seed=7)[0].items()}
    result = {"card": card(), "time": time.strftime("%Y-%m-%d %H:%M:%S")}
    for nt in (1000, 4096):
        result["nt%d" % nt] = workload("nt%d" % nt, nt, list(ROUTES), args.reps, hp, dev)
    result["nt1e5"] = workload("nt1e5", 100_000, ["lowrank_diag"], args.reps, hp, dev)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(result, fh, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
