"""Resident partials: incremental evaluation (update_nodes, _calculate_partials treelikelihood.c:1645-1734) and the single-branch
fast path (_calculate_uppper :2592-2686, calculate_dldt_uppper :2195-2262, d2lnldt2_uppper :2267-2335).

CPU part: the numpy restatement in oracle.branch_derivatives against the reference's own values (tests/golden/branch_derivatives.npz,
made by oracle/make_golden.py from the unmodified reference).  GPU part: the C-ABI entry points against the oracle.
Tolerance: 1e-10 relative on lnL; derivatives relative to max(|d|, 1e-6 * scale) like the branch gradients (tests/util.py).
"""
import os

import numpy as np
import pytest

import physher_b200 as phb
from oracle import oracle as O
from physher_b200 import models, synthetic as syn
from physher_b200.treelikelihood import OPT_INCREMENTAL
from tests.util import GOLDEN, RTOL, grad_err, rel_err


def fixture_problem(tag):
    z = dict(np.load(os.path.join(GOLDEN, "branch_derivatives.npz")))
    g = {k[len(tag) + 1:]: v for k, v in z.items() if k.startswith(tag + "_")}
    pb = O.Problem(left=g["left"], right=g["right"], parent=g["parent"], root=int(g["root"]), nstate=int(g["nstate"]),
                   tip_states=g.get("tip_states"), tip_partials=g.get("tip_partials"), use_tip_states=bool(g["use_tip_states"]),
                   weights=g["weights"], freqs=g["freqs"], rates=g["rates"], props=g["props"], bl=g["bl"], evec=g["evec"], eval=g["eval"],
                   ivec=g["ivec"])
    return pb, g


def deriv_err(got, want):
    """columns lnL, d1, d2: lnL relative; derivatives relative to max(|d|, 1e-6 * column max)"""
    got, want = np.atleast_2d(got), np.atleast_2d(want)
    e = np.max(np.abs(got[:, 0] - want[:, 0]) / np.abs(want[:, 0]))
    for q in (1, 2):
        e = max(e, grad_err(got[:, q], want[:, q]))
    return e


@pytest.mark.parametrize("tag", ["g4", "c1"])
def test_oracle_branch_derivatives_pinned_on_reference(tag):
    pb, g = fixture_problem(tag)
    for i, n in enumerate(g["nodes"]):
        got = O.branch_derivatives(pb, int(n), g["bl"][n] * g["factors"])
        assert np.max(np.abs(got - g["ref_branch"][i]) / np.abs(g["ref_branch"][i])) < 1e-11
    # at the current length the single-branch lnL is the tree's lnL
    assert rel_err(float(g["ref_branch"][0][1][0]), float(g["ref_lnl"])) < 1e-12


def synthetic_problem(S, T, P, C, seed, tip_states=True, unknown=0.02):
    topo = syn.random_topology(T, seed)
    if S == 4:
        m = models.gtr([0.05, 0.3, 0.1, 0.15, 0.3, 0.1], [0.1, 0.2, 0.3, 0.4])
    else:
        m = models.random_reversible(S, seed + 5)
    rates, props = models.discrete_gamma(0.5, C) if C > 1 else (np.ones(1), np.ones(1))
    st = syn.random_patterns(T, P, S, 0.25, seed + 1, unknown_frac=unknown)
    pb = O.Problem(left=topo.left, right=topo.right, parent=topo.parent, root=topo.root, nstate=S, tip_states=st,
                   weights=np.random.default_rng(seed + 2).integers(1, 4, P).astype(np.float64), freqs=m.freqs, rates=rates, props=props,
                   bl=syn.random_branch_lengths(topo, seed + 3), evec=m.evec, eval=m.eval, ivec=m.ivec)
    if not tip_states:
        part = np.where(st[:, :, None] < S, np.eye(S + 1)[np.minimum(st, S)][:, :, :S], 1.0)
        pb.tip_partials, pb.use_tip_states = part.astype(np.float64), False
    return pb


gpu = pytest.mark.gpu


@gpu
@pytest.mark.parametrize("tag", ["g4", "c1"])
def test_branch_against_reference_values(tag):
    pb, g = fixture_problem(tag)
    tlk = phb.SingleTreeLikelihood.from_problem(pb)
    tlk.update_uppers()
    for i, n in enumerate(g["nodes"]):
        lnl, d1, d2 = tlk.calculate_branch(int(n), g["bl"][n] * g["factors"])
        assert deriv_err(np.stack([lnl, d1, d2], 1), g["ref_branch"][i]) < RTOL
    tlk.close()


@gpu
@pytest.mark.parametrize("S,C,tip_states", [(4, 4, True), (4, 1, False), (20, 4, True), (20, 2, False), (61, 1, True), (5, 3, True)],
                         ids=["nuc4-g4", "nuc4-partials", "aa20-g4", "aa20-partials", "codon61", "generic5"])
def test_branch_all_nodes_against_oracle(S, C, tip_states):
    pb = synthetic_problem(S, 9, 301, C, 40 + S, tip_states)
    tlk = phb.SingleTreeLikelihood.from_problem(pb)
    full = O.evaluate(pb)
    for n in range(pb.nnodes):
        if n == pb.root:
            continue
        cands = pb.bl[n] * np.array([1.0, 0.3, 1.7])
        lnl, d1, d2 = tlk.calculate_branch(n, cands)
        want = O.branch_derivatives(pb, n, cands)
        assert deriv_err(np.stack([lnl, d1, d2], 1), want) < RTOL, n
        # at the current length: the tree's lnL and this branch's gradient entry
        assert rel_err(lnl[0], full["lnl"]) < RTOL
        if not (pb.unrooted and n == pb.right[pb.root]):
            assert abs(d1[0] - full["grad"][n]) <= RTOL * max(abs(full["grad"][n]), 1e-6 * np.abs(full["grad"]).max())
    tlk.close()


@gpu
@pytest.mark.parametrize("S,C", [(4, 4), (20, 4), (61, 1), (7, 2)], ids=["nuc4", "aa20", "codon61", "generic7"])
def test_incremental_lnl_and_gradient(S, C):
    """a sequence of single-branch changes evaluated incrementally == full evaluations of the same states"""
    pb = synthetic_problem(S, 12, 257, C, 70 + S)
    inc = phb.SingleTreeLikelihood.from_problem(pb)
    inc.set_option(OPT_INCREMENTAL, 1)
    rng = np.random.default_rng(5)
    bl = pb.bl.copy()
    assert rel_err(inc.calculate(), O.evaluate(pb, gradient=False)["lnl"]) < RTOL
    base_launches = inc.launch_count()
    for step in range(6):
        n = int(rng.integers(0, pb.nnodes))
        if n == pb.root:
            continue
        bl[n] *= float(rng.uniform(0.5, 2.0))
        inc.set_branch_length(n, bl[n])
        if step % 3 == 2:  # two branches at once
            m = (n + 3) % pb.nnodes
            if m != pb.root:
                bl[m] *= 1.3
                inc.set_branch_length(m, bl[m])
        pb.bl = bl.copy()
        want = O.evaluate(pb)
        before = inc.launch_count()
        assert rel_err(inc.calculate(), want["lnl"]) < RTOL
        assert inc.launch_count() - before < 3 * 12 + 8  # a handful of ancestors, not the whole tree
        if step % 2 == 1:
            assert grad_err(inc.gradient(), want["grad"]) < RTOL
    # whole-vector update: only the branches that differ are recomputed
    bl2 = bl.copy()
    bl2[1] *= 0.7
    pb.bl = bl2
    inc.set_branch_lengths(bl2)
    want = O.evaluate(pb)
    assert rel_err(inc.calculate(), want["lnl"]) < RTOL
    assert grad_err(inc.gradient(), want["grad"]) < RTOL
    assert inc.launch_count() > base_launches
    inc.close()


@gpu
def test_branch_optimisation_walk():
    """the access pattern of serial_brent_optimize_tree (optimizer.c:111-152): visit branches in post-order, evaluate candidates
    through the fast path, keep the best, move on -- lnL after every kept change equals a full evaluation"""
    pb = synthetic_problem(4, 10, 200, 4, 91)
    tlk = phb.SingleTreeLikelihood.from_problem(pb)
    tlk.update_uppers()
    bl = pb.bl.copy()
    for n in range(pb.nnodes):
        if n == pb.root or n == pb.right[pb.root]:
            continue
        cands = bl[n] * np.array([0.5, 0.8, 1.0, 1.25, 2.0])
        lnl, d1, d2 = tlk.calculate_branch(n, cands)
        k = int(np.argmax(lnl))
        bl[n] = cands[k]
        tlk.set_branch_length(n, bl[n])
        pb.bl = bl.copy()
        assert rel_err(lnl[k], O.evaluate(pb, gradient=False)["lnl"]) < RTOL
        assert rel_err(tlk.calculate(), lnl[k]) < RTOL
    tlk.close()


@gpu
@pytest.mark.parametrize("S,C", [(4, 4), (20, 2)], ids=["nuc4", "aa20"])
def test_branch_under_rescaling(S, C):
    """scaled partials: the single-branch lnL at the current length is the tree's lnL, its derivative the gradient entry, and
    both agree with the unscaled oracle (the log factors of U_n and L_n are added back)"""
    pb = synthetic_problem(S, 10, 120, C, 17 + S)
    tlk = phb.SingleTreeLikelihood.from_problem(pb)
    tlk.set_option(phb.treelikelihood.OPT_SCALING_THRESHOLD_EXP, 2)  # 1e-2: scaling actually fires on this small tree
    tlk.use_rescaling(True)
    full = O.evaluate(pb)
    for n in (0, 4, pb.ntips + 1, pb.ntips + 4):
        if n == pb.root:
            continue
        cands = pb.bl[n] * np.array([1.0, 2.0])
        lnl, d1, d2 = tlk.calculate_branch(n, cands)
        want = O.branch_derivatives(pb, n, cands)
        assert deriv_err(np.stack([lnl, d1, d2], 1), want) < 1e-9
        assert rel_err(lnl[0], full["lnl"]) < 1e-9
    tlk.close()


@gpu
def test_branch_candidates_past_one_launch():
    """70,000 candidate lengths in one call: the values of the same lengths scored in slices of at most 65,535, and one more score
    launch than a call whose items fit one grid.y"""
    pb = synthetic_problem(4, 8, 64, 2, 55)
    tlk = phb.SingleTreeLikelihood.from_problem(pb)
    n = next(i for i in range(pb.nnodes) if i != pb.root and pb.left[i] >= 0)
    cands = pb.bl[n] * np.linspace(0.2, 3.0, 70000)
    tlk.calculate_branch(n, cands[:2])

    def run(c):
        before = tlk.launch_count()
        out = np.stack(tlk.calculate_branch(n, c), 1)
        return tlk.launch_count() - before, out

    one, head = run(cands[:65535])
    two, out = run(cands)
    assert two == one + 1
    _, tail = run(cands[65535:])
    assert np.array_equal(out, np.concatenate([head, tail]))
    assert deriv_err(out[::997], O.branch_derivatives(pb, n, cands[::997])) < RTOL
    tlk.close()


@gpu
def test_branch_errors():
    pb = synthetic_problem(4, 6, 50, 1, 3)
    tlk = phb.SingleTreeLikelihood.from_problem(pb)
    with pytest.raises(phb.PhysherB200Error):
        tlk.calculate_branch(pb.root, [0.1])
    with pytest.raises(phb.PhysherB200Error):
        tlk.calculate_branch(0, [-0.1])
    tlk.close()
