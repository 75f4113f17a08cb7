#!/usr/bin/env python
"""Timing of the NNI quintet scores (phb_tlk_nni_quintet_scores) beside the NNI scores and the per-candidate loop they replace, on a
bench.py workload:

    python tools/bench_nni_quintet.py --config c2 [--patterns N] [--reps R] [--loop-moves K]

scratch     update_all_nodes() + nni_quintet_scores(): every move of the unrooted neighbourhood from scratch (resident lowers and uppers
            first)
repeat      nni_quintet_scores(moves, t_five) with new lengths only: the matrix table, the score pass and the sum
kernel      the score pass alone (k_nni_quintet<4> or k_nni_quintet_any), CUDA events over the repeats (PHB_OPT_TIMING); bandwidth on
            the bytes it must read: the four operand partials of every move (8 C S bytes per pattern, 1 byte for a state tip)
nni         the same repeat and score pass of nni_scores(moves, t_central), which gives the central branch only
loop        set_topology(exchanged) + the five lengths + branch_hessian_diagonal() + set_topology(back) and the lengths back over K
            sampled moves on a second object, extrapolated to every move (labelled as such); the largest relative lnL difference
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
from tools.bench_nni import exchanged  # noqa: E402


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

    def sib(x):
        p = parent[x]
        return topo.right[p] if topo.left[p] == x else topo.left[p]

    def five(x, y):
        v = parent[y]
        p = parent[v]
        o = (p if p != topo.root else -1) if parent[x] == p else sib(x)
        return [v, sib(y), x, y, o]

    nodes = np.array([five(int(x), int(y)) for x, y in moves])
    t5 = np.where(nodes >= 0, bl[np.maximum(nodes, 0)], 0.0)
    out["moves"] = n

    def timed(fn, reps):
        fn()  # warm-up
        t0 = time.perf_counter()
        for _ in range(reps):
            r = fn()
        return (time.perf_counter() - t0) * 1e3 / reps, r

    def scratch():
        tlk.update_all_nodes()
        return tlk.nni_quintet_scores(moves)

    out["scratch_ms"], (lnls, grads, hess) = timed(scratch, a.reps)
    rng = np.random.default_rng(5)
    tfs = [t5 * rng.uniform(0.5, 2.0, t5.shape) for _ in range(a.reps + 1)]
    tcs = [t[:, 0].copy() for t in tfs]
    tlk.set_option(OPT_TIMING, 1)
    tlk.nni_quintet_scores(moves)  # the option marks the object for an evaluation; settle it before the timed repeats
    for key, fn, lens in (("", lambda t: tlk.nni_quintet_scores(moves, t), tfs), ("nni_", lambda t: tlk.nni_scores(moves, t), tcs)):
        it = iter(lens)
        k0 = tlk.kernel_time()
        out[key + "repeat_ms"], _ = timed(lambda: fn(next(it)), a.reps)
        k1 = tlk.kernel_time()
        out[key + "kernel_ms"] = (k1[0] - k0[0]) / (a.reps + 1)
        out[key + "kernel_launches_per_call"] = (k1[1] - k0[1]) / (a.reps + 1)
    # bytes the score pass reads: the four operands of every move (U_p an upper partial)
    row = 8 * C * S * P
    nbytes = 0
    for (c, k, x, y, o) in nodes:
        for nd in (k, x, y):
            nbytes += P if nd < T else row
        if o >= 0:
            nbytes += row if parent[x] == parent[c] else (P if o < T else row)
    out["kernel_bytes"] = nbytes
    out["kernel_GBps"] = nbytes / (out["kernel_ms"] * 1e-3) / 1e9
    out["kernel_vs_nni_kernel"] = out["kernel_ms"] / out["nni_kernel_ms"]
    tlk.close()  # the loop's object needs the device memory (resident partials of its own)
    # the loop a caller ran before: per move a topology change, the five lengths and the Hessian diagonal, on its own object
    base = make()
    base.calculate()
    sample = np.sort(rng.choice(n, size=min(a.loop_moves, n), replace=False))
    loop_lnl = np.zeros(len(sample))

    def loop():
        for i, k in enumerate(sample):
            lf, rt = exchanged(topo.left, topo.right, parent, int(moves[k, 0]), int(moves[k, 1]))
            base.set_topology(lf, rt, topo.root)
            base.set_branch_lengths(bl)  # the five lengths (here the current ones)
            loop_lnl[i] = base.branch_hessian_diagonal()[0]
            base.set_topology(topo.left, topo.right, topo.root)
            base.set_branch_lengths(bl)
        return loop_lnl

    loop_ms, _ = timed(loop, 1)
    out["loop_sampled_moves"] = len(sample)
    out["loop_ms_per_move"] = loop_ms / len(sample)
    out["loop_ms_extrapolated_to_all_moves"] = loop_ms / len(sample) * n
    out["speedup_scratch_vs_extrapolated_loop"] = out["loop_ms_extrapolated_to_all_moves"] / out["scratch_ms"]
    out["max_rel_diff_vs_loop"] = float(np.max(np.abs(lnls[sample] - loop_lnl) / np.abs(loop_lnl)))
    out["nonfinite"] = int(np.sum(~np.isfinite(grads)) + np.sum(~np.isfinite(hess)) + np.sum(~np.isfinite(lnls)))
    print(json.dumps(out), flush=True)
    assert out["max_rel_diff_vs_loop"] < 1e-10, out
    base.close()


if __name__ == "__main__":
    main()
