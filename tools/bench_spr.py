#!/usr/bin/env python
"""Timing of the SPR regraft scores (phb_tlk_spr_scores) beside the per-candidate loop they replace, on a bench.py workload:

    python tools/bench_spr.py --config c2 [--patterns N] [--reps R] [--loop-targets K]

Three pruned subtrees per workload: a tip, a cherry and a clade of about T/4 tips, each with every target of the unrooted enumeration.
scratch     update_all_nodes() + spr_scores(s): lowers made resident, the pruned pass, the matrix table, the score pass and the sum
repeat      spr_scores(s, targets, t_pendant) with new pendant lengths (the pruned pass runs again: the call leaves the current tree's
            path lowers marked for recomputation)
kernel      the score pass alone (k_spr_score<4> or k_spr_score_any), CUDA events over the repeats (PHB_OPT_TIMING); bandwidth on the
            bytes it must read: U~_e and L~_e of every target (8 C S bytes per pattern each, 1 byte for a state tip) -- L_s, the same
            for every target, is counted once
loop        set_topology(regrafted) + calculate() + set_topology(back) over K sampled targets on a second object, extrapolated to every
            target (labelled as such); the largest relative lnL difference between the two on the sampled targets
Wall-clock around synchronous C-ABI calls, after a warm-up call of each; one JSON line per workload with the card's name and power limit.
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
import physher_b200 as phb  # noqa: E402
from physher_b200.treelikelihood import OPT_TIMING  # noqa: E402
from tools.bench_hessian import card  # noqa: E402


def regrafted(left, right, parent, s, e):
    """child arrays of the tree with the subtree of s pruned (with p = parent[s]) and regrafted on the branch above e"""
    left, right, parent = left.copy(), right.copy(), parent.copy()
    p = parent[s]
    g = parent[p]
    b = right[p] if left[p] == s else left[p]
    for arr in (left, right):
        if arr[g] == p:
            arr[g] = b
    parent[b] = g
    h = parent[e]
    for arr in (left, right):
        if arr[h] == e:
            arr[h] = p
    if left[p] == s:
        right[p] = e
    else:
        left[p] = e
    return left, right


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="c2", choices=sorted(bench.CONFIGS))
    ap.add_argument("--patterns", type=int, default=0)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--loop-targets", type=int, default=8)
    a = ap.parse_args()
    cfg = dict(bench.CONFIGS[a.config])
    if a.patterns:
        cfg["patterns"] = a.patterns
    topo, bl, m, rates, props, patterns, weights = bench.make_inputs(cfg, 0)
    T, P, S, C = cfg["taxa"], cfg["patterns"], cfg["states"], cfg["cats"]
    N = 2 * T - 1

    def make():
        tlk = phb.SingleTreeLikelihood(topo.left, topo.right, topo.root, S, C, P, use_tip_states=True, device=0)
        tlk.set_tip_states(patterns)
        tlk.set_pattern_weights(weights)
        tlk.set_eigen(m.evec, m.eval, m.ivec)
        tlk.set_frequencies(m.freqs)
        tlk.set_site_model(rates, props)
        tlk.set_branch_lengths(bl)
        return tlk

    parent = np.full(N, -1)
    for v in range(N):
        for c in (topo.left[v], topo.right[v]):
            if c >= 0:
                parent[c] = v
    tips = np.zeros(N, dtype=np.int64)
    for v in range(N):  # tips below each node
        if topo.left[v] < 0:
            u = v
            while u >= 0:
                tips[u] += 1
                u = parent[u]
    prunable = [n for n in range(N) if n != topo.root and parent[n] != topo.root]
    choices = {
        "tip": next(n for n in prunable if topo.left[n] < 0),
        "cherry": next(n for n in prunable if topo.left[n] >= 0 and tips[n] == 2),
        "clade": min((n for n in prunable if topo.left[n] >= 0), key=lambda n: abs(tips[n] - T / 4)),
    }

    def timed(fn, reps):
        fn()  # warm-up
        t0 = time.perf_counter()
        for _ in range(reps):
            r = fn()
        return (time.perf_counter() - t0) * 1e3 / reps, r

    tlk = make()
    base = make()
    base.calculate()
    name, power = card()
    out = {"config": bench.workload_name(cfg), "nodes": N, "gpu": name, "power_limit": power, "subtrees": []}
    rng = np.random.default_rng(5)
    row = 8 * C * S * P
    for kind, s in choices.items():
        rec = {"kind": kind, "s": int(s), "tips_below_s": int(tips[s])}
        targets = tlk.spr_targets(s)
        n = len(targets)
        rec["targets"] = n

        def scratch():
            tlk.update_all_nodes()
            return tlk.spr_scores(s, targets)

        rec["scratch_ms"], (lnl, scores) = timed(scratch, a.reps)
        tps = [bl[s] * rng.uniform(0.5, 2.0, n) for _ in range(a.reps + 1)]
        it = iter(tps)
        tlk.set_option(OPT_TIMING, 1)
        tlk.spr_scores(s, targets)  # the option marks the object for an evaluation; settle it before the timed repeats
        k0 = tlk.kernel_time()
        rec["repeat_ms"], _ = timed(lambda: tlk.spr_scores(s, targets, next(it)), a.reps)
        k1 = tlk.kernel_time()
        tlk.set_option(OPT_TIMING, 0)
        rec["kernel_ms"] = (k1[0] - k0[0]) / (a.reps + 1)
        rec["kernel_launches_per_call"] = (k1[1] - k0[1]) / (a.reps + 1)
        nbytes = (P if s < T else row) + sum(row + (P if e < T else row) for e in targets)
        rec["kernel_bytes"] = int(nbytes)
        rec["kernel_GBps"] = nbytes / (rec["kernel_ms"] * 1e-3) / 1e9
        # the loop a caller ran before: one topology change and one evaluation per candidate, on its own object
        sample = np.sort(rng.choice(n, size=min(a.loop_targets, n), replace=False))
        loop_lnl = np.zeros(len(sample))

        def loop():
            for i, k in enumerate(sample):
                lf, rt = regrafted(topo.left, topo.right, parent, int(s), int(targets[k]))
                base.set_topology(lf, rt, topo.root)
                loop_lnl[i] = base.calculate()
                base.set_topology(topo.left, topo.right, topo.root)
            return loop_lnl

        loop_ms, _ = timed(loop, 1)
        rec["loop_sampled_targets"] = len(sample)
        rec["loop_ms_per_target"] = loop_ms / len(sample)
        rec["loop_ms_extrapolated_to_all_targets"] = loop_ms / len(sample) * n
        rec["speedup_scratch_vs_extrapolated_loop"] = rec["loop_ms_extrapolated_to_all_targets"] / rec["scratch_ms"]
        rec["max_rel_diff_vs_loop"] = float(np.max(np.abs(scores[sample, 0] - loop_lnl) / np.abs(loop_lnl)))
        rec["lnl"] = lnl
        rec["nonfinite"] = int(np.sum(~np.isfinite(scores)))
        out["subtrees"].append(rec)
    print(json.dumps(out), flush=True)
    assert all(r["max_rel_diff_vs_loop"] < 1e-10 for r in out["subtrees"]), out
    tlk.close()
    base.close()


if __name__ == "__main__":
    main()
