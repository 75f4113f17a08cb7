#!/usr/bin/env python
"""Timing of the SPR tripod scores (phb_tlk_spr_tripod_scores) beside the SPR scores on the same subtree and the per-candidate loop they
replace, on a bench.py workload:

    python tools/bench_spr_tripod.py --config c2 [--patterns N] [--reps R] [--loop-targets K]

Three pruned subtrees per workload: a tip, a cherry and a clade of about T/4 tips, each with every target of the unrooted enumeration.
scratch     update_all_nodes() + spr_tripod_scores(s): lowers made resident, the pruned pass with b's branch joined (b's matrix rebuilt
            at the joined length and every matrix back at the current lengths after it), the matrix table, the score pass and the sum
repeat      spr_tripod_scores(s, targets, t_tripod) with new tripod lengths
kernel      the score pass alone (k_spr_tripod<4> or k_spr_tripod_any), CUDA events over the repeats (PHB_OPT_TIMING); bandwidth on the
            bytes it must read, the model of tools/bench_spr.py (the operands are the same: U~_e and L~_e of every target, 8 C S bytes
            per pattern each, 1 byte for a state tip; L_s counted once)
spr         the same three figures for spr_scores(s) in the same process: the five-matrix contraction next to the nine-matrix one
loop        set_topology(regrafted) + set_branch_lengths(tripod, joined b) + calculate() over K sampled targets on a second object,
            extrapolated to every target (labelled as such); the largest relative lnL difference between the two on the sampled targets
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
from tools.bench_spr import regrafted  # noqa: E402


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

    def kernel_timed(fn, reps):
        tlk.set_option(OPT_TIMING, 1)
        fn()  # the option marks the object for an evaluation; settle it before the timed repeats
        k0 = tlk.kernel_time()
        ms, _ = timed(fn, reps)
        k1 = tlk.kernel_time()
        tlk.set_option(OPT_TIMING, 0)
        return ms, (k1[0] - k0[0]) / (reps + 1), (k1[1] - k0[1]) / (reps + 1)

    tlk = make()
    base = make()
    base.calculate()
    name, power = card()
    out = {"config": bench.workload_name(cfg), "nodes": N, "gpu": name, "power_limit": power, "subtrees": []}
    rng = np.random.default_rng(5)
    row = 8 * C * S * P
    for kind, s in choices.items():
        p = int(parent[s])
        b = int(topo.right[p] if topo.left[p] == s else topo.left[p])
        rec = {"kind": kind, "s": int(s), "tips_below_s": int(tips[s])}
        targets = tlk.spr_targets(s)
        n = len(targets)
        rec["targets"] = n
        lb = bl[b] + bl[p]
        half = np.array([(lb if e == b else bl[e]) / 2 for e in targets])
        tri0 = np.column_stack([half, half, np.full(n, bl[s])])

        def scratch():
            tlk.update_all_nodes()
            return tlk.spr_tripod_scores(s, targets)

        rec["scratch_ms"], (lnl, grad, hess) = timed(scratch, a.reps)
        tris = [tri0 * rng.uniform(0.5, 2.0, tri0.shape) for _ in range(a.reps + 2)]
        it = iter(tris)
        rec["repeat_ms"], rec["kernel_ms"], rec["kernel_launches_per_call"] = kernel_timed(lambda: tlk.spr_tripod_scores(s, targets, next(it)),
                                                                                           a.reps)
        nbytes = (P if s < T else row) + sum(row + (P if e < T else row) for e in targets)
        rec["kernel_bytes"] = int(nbytes)
        rec["kernel_GBps"] = nbytes / (rec["kernel_ms"] * 1e-3) / 1e9

        def spr_scratch():
            tlk.update_all_nodes()
            return tlk.spr_scores(s, targets)

        rec["spr_scratch_ms"], _ = timed(spr_scratch, a.reps)
        rec["spr_repeat_ms"], rec["spr_kernel_ms"], _ = kernel_timed(lambda: tlk.spr_scores(s, targets), a.reps)
        rec["kernel_ratio_tripod_vs_spr"] = rec["kernel_ms"] / rec["spr_kernel_ms"]
        # the loop a caller ran before: one topology change, the tripod lengths and one evaluation per candidate, on its own object
        sample = np.sort(rng.choice(n, size=min(a.loop_targets, n), replace=False))
        loop_lnl = np.zeros(len(sample))

        def loop():
            for i, k in enumerate(sample):
                e = int(targets[k])
                lf, rt = regrafted(topo.left, topo.right, parent, int(s), e)
                lens = bl.copy()
                lens[b] = lb
                lens[p], lens[e], lens[s] = tri0[k]
                base.set_topology(lf, rt, topo.root)
                base.set_branch_lengths(lens)
                loop_lnl[i] = base.calculate()
                base.set_topology(topo.left, topo.right, topo.root)
                base.set_branch_lengths(bl)
            return loop_lnl

        loop_ms, _ = timed(loop, 1)
        rec["loop_sampled_targets"] = len(sample)
        rec["loop_ms_per_target"] = loop_ms / len(sample)
        rec["loop_ms_extrapolated_to_all_targets"] = loop_ms / len(sample) * n
        rec["speedup_scratch_vs_extrapolated_loop"] = rec["loop_ms_extrapolated_to_all_targets"] / rec["scratch_ms"]
        rec["max_rel_diff_vs_loop"] = float(np.max(np.abs(lnl[sample] - loop_lnl) / np.abs(loop_lnl)))
        rec["nonfinite"] = int(np.sum(~np.isfinite(grad)) + np.sum(~np.isfinite(hess)) + np.sum(~np.isfinite(lnl)))
        out["subtrees"].append(rec)
    print(json.dumps(out), flush=True)
    assert all(r["max_rel_diff_vs_loop"] < 1e-10 for r in out["subtrees"]), out
    tlk.close()
    base.close()


if __name__ == "__main__":
    main()
