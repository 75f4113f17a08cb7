#!/usr/bin/env python
"""Timing of the branch-length Hessian diagonal (phb_tlk_branch_hessian_diagonal) beside one gradient evaluation and beside the
single-branch loop it replaces, on a bench.py workload:

    python tools/bench_hessian.py --config c2 [--patterns N] [--reps R]

gradient    update_all_nodes() + gradient(): one lnL + gradient evaluation from scratch (the bench.py step)
hessian     update_all_nodes() + branch_hessian_diagonal(): lnL, gradient and Hessian diagonal from scratch
uppers      update_all_nodes() + update_uppers(): the part of the loop (and of the resident-partials route) before any branch term
loop        update_all_nodes() + update_uppers() + one calculate_branch(n, [t_n]) per branch: what a caller paid before
Wall-clock around synchronous C-ABI calls (each returns its result to the host), after one warm-up call of each; one JSON line
with the card's name and power limit.  The two diagonals must agree within 1e-10 (grad_err convention of tests/util.py), the
gradient of the call with gradient() within GRAD_TOL.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
import physher_b200 as phb  # noqa: E402
from tests.util import FLOOR_LARGE, RTOL, grad_err  # noqa: E402


# The gradient of the call against gradient(): on the resident route two kernel families (single-branch kernels against the
# tensor-core gradient) sum a full-size alignment in different orders; at 61 states and 250k patterns they differ by 2e-10
# (NVIDIA B200), within what the reordering of 250k terms of both signs gives.  The diagonals come from the same kernels and
# must agree within RTOL.
GRAD_TOL = 1e-9


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=30).stdout.strip().splitlines()
        name, power = (s.strip() for s in out[0].split(","))
        return name, power
    except Exception as exc:  # the numbers are still worth having; say why the card is not named
        return f"unknown ({exc!r})", "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="c2", choices=sorted(bench.CONFIGS))
    ap.add_argument("--patterns", type=int, default=0)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--loop-reps", type=int, default=1)
    a = ap.parse_args()
    cfg = dict(bench.CONFIGS[a.config])
    if a.patterns:
        cfg["patterns"] = a.patterns
    topo, bl, m, rates, props, patterns, weights = bench.make_inputs(cfg, 0)
    T, P, S, C = cfg["taxa"], cfg["patterns"], cfg["states"], cfg["cats"]
    N = 2 * T - 1
    tlk = phb.SingleTreeLikelihood(topo.left, topo.right, topo.root, S, C, P, use_tip_states=True, device=0)
    tlk.set_tip_states(patterns)
    tlk.set_pattern_weights(weights)
    tlk.set_eigen(m.evec, m.eval, m.ivec)
    tlk.set_frequencies(m.freqs)
    tlk.set_site_model(rates, props)
    tlk.set_branch_lengths(bl)
    name, power = card()
    out = {"config": bench.workload_name(cfg), "nodes": N, "gpu": name, "power_limit": power}

    def timed(fn, reps):
        fn()  # warm-up
        t0 = time.perf_counter()
        for _ in range(reps):
            r = fn()
        return (time.perf_counter() - t0) * 1e3 / reps, r

    def gradient():
        tlk.update_all_nodes()
        return tlk.gradient()

    def hessian():
        tlk.update_all_nodes()
        return tlk.branch_hessian_diagonal()

    branches = [n for n in range(N) if n != topo.root]

    def loop():
        tlk.update_all_nodes()
        tlk.update_uppers()
        h = np.zeros(N)
        for n in branches:
            h[n] = tlk.calculate_branch(n, [bl[n]])[2][0]
        if tlk.right[topo.root] >= 0:  # the unrooted convention (PHB_OPT_UNROOTED, on by default)
            h[topo.right[topo.root]] = 0.0
        return h

    out["gradient_ms"], g = timed(gradient, a.reps)
    out["hessian_ms"], (lnl, gh, hess) = timed(hessian, a.reps)
    out["hessian_kernels"] = tlk.last_kernels()  # 2: fused 4-state walk; otherwise the resident-partials route
    out["uppers_ms"], _ = timed(lambda: (tlk.update_all_nodes(), tlk.update_uppers()), a.reps)
    out["loop_ms"], hloop = timed(loop, a.loop_reps)
    out["loop_launches_per_branch"] = 3
    out["hessian_over_gradient"] = out["hessian_ms"] / out["gradient_ms"]
    out["loop_over_hessian"] = out["loop_ms"] / out["hessian_ms"]
    # two different kernel families over a full-size alignment: entries that nearly cancel carry the noise of the pattern order
    # (tests/util.py, FLOOR_LARGE)
    out["grad_err_vs_gradient"] = grad_err(gh, g, FLOOR_LARGE)
    out["hess_err_vs_loop"] = grad_err(hess, hloop)
    out["lnl"] = lnl
    out["nonfinite"] = {"hessian": int(np.sum(~np.isfinite(hess))), "loop": int(np.sum(~np.isfinite(hloop)))}
    if not out["hess_err_vs_loop"] < RTOL:  # where the two disagree
        bad = np.argsort(-np.nan_to_num(np.abs(hess - hloop), nan=np.inf))[:5]
        out["worst"] = [(int(n), float(hess[n]), float(hloop[n]), int(n < T)) for n in bad]
    print(json.dumps(out), flush=True)
    assert out["hess_err_vs_loop"] < RTOL, out
    assert out["grad_err_vs_gradient"] < GRAD_TOL, out
    tlk.close()


if __name__ == "__main__":
    main()
