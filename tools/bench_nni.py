#!/usr/bin/env python
"""Timing of the NNI neighbourhood scores (phb_tlk_nni_scores) beside the per-candidate loop they replace, on a bench.py workload:

    python tools/bench_nni.py --config c2 [--patterns N] [--reps R] [--loop-moves K]

scratch     update_all_nodes() + nni_scores(): every move of the unrooted neighbourhood from scratch (resident lowers and uppers first)
repeat      nni_scores(moves, t_central) with new central lengths only: the matrix table, the score pass and the sum
kernel      the score pass alone (k_nni_score<4>, or k_nni_operands + k_nni_contract), CUDA events over the repeats (PHB_OPT_TIMING);
            bandwidth on the bytes it must read: each operand partial of a (v, x) group once (8 C S bytes per pattern, 1 byte for a
            state tip), plus the operand scratch the route for other state counts writes and reads back
loop        set_topology(exchanged) + calculate() + set_topology(back) over K sampled moves on a second object, extrapolated to every
            move (labelled as such); the largest relative lnL difference between the two on the sampled moves
Wall-clock around synchronous C-ABI calls, after a warm-up call of each; one JSON line with the card's name and power limit.
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


def exchanged(left, right, parent, x, y):
    left, right = left.copy(), right.copy()
    v, u = parent[y], parent[x]
    if left[v] == y:
        left[v] = x
    else:
        right[v] = x
    if left[u] == x:
        left[u] = y
    else:
        right[u] = y
    return left, right


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="c2", choices=sorted(bench.CONFIGS))
    ap.add_argument("--patterns", type=int, default=0)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--loop-moves", type=int, default=8)
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

    tlk = make()
    name, power = card()
    out = {"config": bench.workload_name(cfg), "nodes": N, "gpu": name, "power_limit": power}
    moves = tlk.nni_moves()
    n = len(moves)
    parent = np.full(N, -1)
    for v in range(N):
        for c in (topo.left[v], topo.right[v]):
            if c >= 0:
                parent[c] = v
    out["moves"] = n

    def timed(fn, reps):
        fn()  # warm-up
        t0 = time.perf_counter()
        for _ in range(reps):
            r = fn()
        return (time.perf_counter() - t0) * 1e3 / reps, r

    def scratch():
        tlk.update_all_nodes()
        return tlk.nni_scores(moves)

    out["scratch_ms"], (lnl, scores) = timed(scratch, a.reps)
    rng = np.random.default_rng(5)
    tcs = [bl[parent[moves[:, 1]]] * rng.uniform(0.5, 2.0, n) for _ in range(a.reps + 1)]
    it = iter(tcs)
    tlk.set_option(OPT_TIMING, 1)
    tlk.nni_scores(moves)  # the option marks the object for an evaluation; settle it before the timed repeats
    k0 = tlk.kernel_time()
    out["repeat_ms"], _ = timed(lambda: tlk.nni_scores(moves, next(it)), a.reps)
    k1 = tlk.kernel_time()
    out["kernel_ms"] = (k1[0] - k0[0]) / (a.reps + 1)
    out["kernel_launches_per_call"] = (k1[1] - k0[1]) / (a.reps + 1)
    # bytes the score pass reads: each operand of a (v, x) group once
    row = 8 * C * S * P

    def operand_bytes(node, upper=False):
        return P if (node < T and not upper) else row

    groups = {}
    for x, y in moves:
        groups.setdefault((int(parent[y]), int(x)), []).append(int(y))
    nbytes = 0
    for (v, x), ys in groups.items():
        p = parent[v]
        nbytes += operand_bytes(x) + operand_bytes(topo.left[v]) + operand_bytes(topo.right[v])
        if parent[x] == p and p != topo.root:
            nbytes += row  # U_p
        elif parent[x] != p:
            w = parent[x]
            nbytes += operand_bytes(topo.left[w] if topo.right[w] == x else topo.right[w])
    if S != 4:
        nbytes += n * 2 * 2 * row  # operand scratch written and read back
    out["kernel_bytes"] = nbytes
    out["kernel_GBps"] = nbytes / (out["kernel_ms"] * 1e-3) / 1e9
    # the loop a caller ran before: one topology change and one evaluation per candidate, on its own object
    base = make()
    base.calculate()
    sample = np.sort(rng.choice(n, size=min(a.loop_moves, n), replace=False))
    loop_lnl = np.zeros(len(sample))

    def loop():
        for i, k in enumerate(sample):
            lf, rt = exchanged(topo.left, topo.right, parent, int(moves[k, 0]), int(moves[k, 1]))
            base.set_topology(lf, rt, topo.root)
            loop_lnl[i] = base.calculate()
            base.set_topology(topo.left, topo.right, topo.root)
        return loop_lnl

    loop_ms, _ = timed(loop, 1)
    out["loop_sampled_moves"] = len(sample)
    out["loop_ms_per_move"] = loop_ms / len(sample)
    out["loop_ms_extrapolated_to_all_moves"] = loop_ms / len(sample) * n
    out["speedup_scratch_vs_extrapolated_loop"] = out["loop_ms_extrapolated_to_all_moves"] / out["scratch_ms"]
    out["max_rel_diff_vs_loop"] = float(np.max(np.abs(scores[sample, 0] - loop_lnl) / np.abs(loop_lnl)))
    out["lnl"] = lnl
    out["nonfinite"] = int(np.sum(~np.isfinite(scores)))
    print(json.dumps(out), flush=True)
    assert out["max_rel_diff_vs_loop"] < 1e-10, out
    tlk.close()
    base.close()


if __name__ == "__main__":
    main()
