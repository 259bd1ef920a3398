"""Throughput of log_likelihood(method="lowrank") against the dense conditional path (DESIGN.md 4.6).

    python scripts/bench_lowrank.py [--out FILE] [--reps N]

Writes one JSON file with the card name and power limit.  The two methods are timed alternately in the
same process with CUDA events around whole calls (Ylm moments included: a new process object per call)
and per-stage CUDA events (StarryProcess._stage_ms).  Workloads:
  long_baseline   B = 512, nt = 4096, conditional, limb-darkened: bench.py's long_baseline_nt4096 inputs
  bench_draws     B = 4096, nt = 1000, normalised: the bench draws (seed 1234)
  incl_grid       calibrate.inclination_log_prob, 10 light curves x 100 samples x 100 inclinations, nt = 1000
  nt1e5           B = 4096, nt = 1e5, normalised (low-rank only: one dense K would take 80 GB)
  cov_stage       the B_inc Sigma product of the covariance stage alone (spb_gemm_nt, same shapes), B = 4096:
                  achieved HBM bandwidth for the 512 KB of Sigma each element reads
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
import starry_process_b200 as spb  # noqa: E402
from starry_process_b200 import _lib, calibrate  # noqa: E402
from starry_process_b200.sp import _ptr, _stream  # noqa: E402

U_LD = [0.4, 0.26]


def card():
    out = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout
        out["power_limit"], out["sm_max_clock"] = [s.strip() for s in q.strip().split(",")]
    except Exception as e:  # noqa: BLE001
        out["power_limit"] = "unavailable (%s)" % e
    return out


def timed(fn):
    """One call: (ms between CUDA events, per-stage ms, result)."""
    stage = {}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    res = fn(stage)
    e1.record()
    torch.cuda.synchronize()
    st = {k: sum(a.elapsed_time(b) for a, b in v) for k, v in stage.items()}
    return e0.elapsed_time(e1), st, res


def compare(name, n_elems, make, reps, methods=("dense", "lowrank")):
    """Alternate the methods `reps` times after one warm-up call each."""
    res = {"elements": n_elems}
    out = {}
    times = {m: [] for m in methods}
    stages = {m: {} for m in methods}
    for r in range(reps + 1):
        for m in methods:
            ms, st, ll = timed(lambda stage, m=m: make(m, stage))
            out[m] = ll
            if r > 0:
                times[m].append(ms)
                for k, v in st.items():
                    stages[m].setdefault(k, []).append(v)
    for m in methods:
        med = float(np.median(times[m]))
        res[m] = {"ms": times[m], "median_ms": med, "evals_per_s": n_elems / med * 1e3,
                  "stage_median_ms": {k: float(np.median(v)) for k, v in stages[m].items()}}
    if len(methods) == 2:
        a, b = out["lowrank"].cpu().numpy().ravel(), out["dense"].cpu().numpy().ravel()
        fin = np.isfinite(b)
        res["same_neginf_pattern"] = bool(np.array_equal(np.isneginf(a), np.isneginf(b)))
        res["max_rel_diff_lowrank_vs_dense"] = float(np.max(np.abs(a[fin] - b[fin]) / np.abs(b[fin])))
    print(name, json.dumps(res), flush=True)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="bench_lowrank.json", help="JSON result file (default: ./bench_lowrank.json)")
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_lowrank.py measures on a CUDA device; none is available")
    dev = torch.device("cuda", 0)
    result = {"card": card(), "time": time.strftime("%Y-%m-%d %H:%M:%S")}

    # long baseline: bench.py long_baseline_phase inputs
    lb = np.load(os.path.join(ROOT, "tests", "golden", "longbaseline_nt4096.npz"))
    r2 = np.load(os.path.join(ROOT, "tests", "golden", "longbaseline_nt4096_r2.npz"))
    B, ns = 512, len(r2["r"])
    rng = np.random.default_rng(41)
    hp = {k: np.concatenate([r2[k], rng.uniform(bench.PRIORS["narrow"][k][0], bench.PRIORS["narrow"][k][1],
                                                B - ns)]) for k in ("r", "c", "n", "mu", "sigma")}
    hd = {k: torch.tensor(v, device=dev) for k, v in hp.items()}
    td, fd = torch.tensor(lb["t"], device=dev), torch.tensor(lb["flux"], device=dev)
    bvar = torch.zeros(B, dtype=torch.float64, device=dev)
    bvar[:ns] = torch.tensor(r2["baseline_var"], device=dev)

    def long_baseline(method, stage):
        gp = spb.StarryProcess(marginalize_over_inclination=False, normalized=False, **hd)
        gp._stage_ms = stage
        return gp.log_likelihood(td, fd, 1e-6, i=60.0, p=1.0, u=U_LD, baseline_var=bvar, method=method)

    result["long_baseline"] = compare("long_baseline", B, long_baseline, args.reps)

    # bench draws, normalised, nt = 1000
    hpb, tb, fb, _ = bench.synthetic_inputs(4096, seed=1234)
    hbd = {k: torch.tensor(v, device=dev) for k, v in hpb.items()}
    tbd, fbd = torch.tensor(tb, device=dev), torch.tensor(fb, device=dev)

    def draws(method, stage):
        gp = spb.StarryProcess(marginalize_over_inclination=False, normalized=True, **hbd)
        gp._stage_ms = stage
        return gp.log_likelihood(tbd, fbd, 1e-6, i=60.0, p=1.0, u=U_LD, method=method)

    result["bench_draws"] = compare("bench_draws", 4096, draws, args.reps)

    # inclination grid, 10 x 100 x 100 at nt = 1000
    a, b = spb.gauss2beta(torch.tensor(hpb["mu"][:100]), torch.tensor(hpb["sigma"][:100]))
    samples = np.stack([hpb["r"][:100], a.numpy(), b.numpy(), hpb["c"][:100], hpb["n"][:100]], axis=1)
    flc = 1e-3 * np.random.default_rng(3).standard_normal((10, len(tb)))
    inc = np.linspace(0.0, 90.0, 100)

    def grid(method, stage):
        return calibrate.inclination_log_prob(tb, flc, samples, inc, ferr=1e-3, p=1.0, u=U_LD, method=method)

    result["incl_grid"] = compare("incl_grid", 10 * 100 * 100, grid, max(1, args.reps - 2))

    # nt = 1e5, low-rank only
    nt = 100_000
    t5 = torch.linspace(0, 90.0, nt, dtype=torch.float64, device=dev)
    f5 = 1e-3 * torch.randn(nt, dtype=torch.float64, device=dev, generator=torch.Generator(device=dev).manual_seed(5))
    hp5 = {k: torch.tensor(v, device=dev) for k, v in bench.synthetic_inputs(4096, seed=7)[0].items()}

    def long_lc(method, stage):
        gp = spb.StarryProcess(marginalize_over_inclination=False, normalized=True, **hp5)
        gp._stage_ms = stage
        return gp.log_likelihood(t5, f5, 1e-6, i=60.0, p=1.0, u=U_LD, method=method)

    torch.cuda.reset_peak_memory_stats()
    result["nt1e5"] = compare("nt1e5", 4096, long_lc, args.reps, methods=("lowrank",))
    result["nt1e5"]["peak_allocated_GB"] = torch.cuda.max_memory_allocated() / 1e9

    # covariance stage: T = B_inc Sigma for 512-element chunks (the chunk the library uses), B = 4096
    ctx = spb.get_context()
    lib, h = ctx.lib, ctx.handle
    Bc = 512
    cov = torch.randn(4096, 256, 256, dtype=torch.float64, device=dev)
    binc = torch.randn(32, 256, dtype=torch.float64, device=dev)
    T = torch.empty(Bc, 32, 256, dtype=torch.float64, device=dev)

    def stage_c():
        for b0 in range(0, 4096, Bc):
            _lib.check(lib.spb_gemm_nt(h, Bc, 32, 256, 256, 1.0, _ptr(binc), 256, 0, _ptr(cov[b0:]), 256, 65536,
                                       0.0, _ptr(T), 256, 32 * 256, _stream()))

    stage_c()
    ts = []
    for _ in range(10):
        ms, _, _ = timed(lambda stage: stage_c())
        ts.append(ms)
    med = float(np.median(ts))
    result["cov_stage"] = {"elements": 4096, "median_ms": med, "bytes_read": 4096 * 65536 * 8,
                           "achieved_TB_per_s": 4096 * 65536 * 8 / (med * 1e-3) / 1e12,
                           "note": "Sigma (2.1 GB) exceeds the 126 MB L2: read from HBM"}
    print("cov_stage", json.dumps(result["cov_stage"]), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(result, fh, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
