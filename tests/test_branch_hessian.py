"""Diagonal of the branch-length Hessian in one call (phb_tlk_branch_hessian_diagonal): d2lnldt2_uppper (treelikelihood.c:2267-2335)
of every branch at its current length, with lnL and the gradient of the same pass.

Route 1 is the fused 4-state walk (GRAD = 3 variant of k_nuc4_walk), route 2 the single-branch kernels over the list of every
non-root node on resident partials (any state count, rescaling, and whatever the walk declines).  Reference values: the unmodified
reference's own d2lnldt2_uppper (tests/golden/branch_derivatives.npz) and the numpy restatement in oracle.branch_derivatives; an
independent check by central differences of the gradient.  Tolerance: RTOL with the grad_err convention of tests/util.py.
"""
import numpy as np
import pytest

import physher_b200 as phb
from oracle import oracle as O
from physher_b200 import models, synthetic as syn
from physher_b200.treelikelihood import (KERNELS_GENERIC, OPT_INCREMENTAL, OPT_SCALING_THRESHOLD_EXP, OPT_UNROOTED, RAN_GENERIC,
                                         RAN_WALK)
from tests.test_branch import fixture_problem, synthetic_problem
from tests.util import RTOL, grad_err, rel_err

gpu = pytest.mark.gpu


def branch_problem(S, T, P, C, seed, tip_states=True):
    """synthetic_problem with every branch of non-zero length and the unrooted convention off: every entry is comparable"""
    pb = synthetic_problem(S, T, P, C, seed, tip_states)
    pb.bl = syn.random_branch_lengths(syn.random_topology(T, seed), seed + 3, unrooted=False)
    pb.unrooted = False
    return pb


def make(pb, kernels=phb.KERNELS_AUTO):
    tlk = phb.SingleTreeLikelihood.from_problem(pb, kernels=kernels)
    tlk.set_option(OPT_UNROOTED, int(pb.unrooted))
    return tlk


def oracle_hessian(pb):
    h = np.zeros(pb.nnodes)
    for n in range(pb.nnodes):
        if n != pb.root:
            h[n] = O.branch_derivatives(pb, n, [pb.bl[n]])[0, 2]
    return h


@gpu
@pytest.mark.parametrize("tag", ["g4", "c1"])
def test_hessian_against_reference_values(tag):
    pb, g = fixture_problem(tag)
    assert g["factors"][1] == 1.0
    tlk = phb.SingleTreeLikelihood.from_problem(pb)
    tlk.set_option(OPT_UNROOTED, 0)
    lnl, grad, hess = tlk.branch_hessian_diagonal()
    nodes = [int(n) for n in g["nodes"]]
    assert grad_err(hess[nodes], np.array([g["ref_branch"][i][1][2] for i in range(len(nodes))])) < RTOL
    assert rel_err(lnl, float(g["ref_lnl"])) < RTOL
    tlk.close()


SHAPES = [  # S, C, tip_states, T, P
    (4, 4, True, 9, 301), (4, 1, False, 9, 301), (20, 4, True, 9, 301), (20, 2, False, 9, 301), (61, 1, True, 9, 301),
    (5, 3, True, 9, 301), (4, 8, True, 9, 301), (4, 4, True, 9, 1), (20, 4, True, 9, 1), (4, 2, True, 2, 301), (4, 4, True, 3, 301),
    (20, 1, True, 3, 77),
]
IDS = ["nuc4-g4", "nuc4-partials", "aa20-g4", "aa20-partials", "codon61", "generic5", "nuc4-c8", "nuc4-p1", "aa20-p1", "nuc4-t2",
       "nuc4-t3", "aa20-t3"]


@gpu
@pytest.mark.parametrize("S,C,tip_states,T,P", SHAPES, ids=IDS)
def test_hessian_every_node_against_oracle(S, C, tip_states, T, P):
    pb = branch_problem(S, T, P, C, 40 + S + T, tip_states)
    tlk = make(pb)
    lnl, grad, hess = tlk.branch_hessian_diagonal()
    full = O.evaluate(pb)
    assert rel_err(lnl, full["lnl"]) < RTOL
    assert grad_err(grad, full["grad"]) < RTOL
    assert hess[pb.root] == 0.0 and grad[pb.root] == 0.0
    assert grad_err(hess, oracle_hessian(pb)) < RTOL
    if S == 4:
        assert tlk.last_kernels() == RAN_WALK
    tlk.close()


@gpu
@pytest.mark.parametrize("C", [1, 4])
def test_hessian_walk_route_and_generic_agree(C):
    """4 states by default run on the fused walk and leave PHB_OPT_INCREMENTAL off; the node-at-a-time route gives the same diagonal"""
    pb = branch_problem(4, 40, 1000, C, 11)
    walk = make(pb)
    lw, gw, hw = walk.branch_hessian_diagonal()
    assert walk.last_kernels() == RAN_WALK
    gen = make(pb, kernels=KERNELS_GENERIC)
    lg, gg, hg = gen.branch_hessian_diagonal()
    assert gen.last_kernels() == RAN_GENERIC
    assert rel_err(lw, lg) < RTOL and grad_err(gw, gg) < RTOL and grad_err(hw, hg) < RTOL
    # the walk route keeps no resident partials: a later length change is a full (fused) evaluation, not an incremental one
    walk.set_branch_length(3, pb.bl[3] * 1.1)
    walk.calculate()
    assert walk.last_kernels() == RAN_WALK
    # with PHB_OPT_INCREMENTAL on, the resident route serves the same values
    walk.set_branch_length(3, pb.bl[3])
    walk.set_option(OPT_INCREMENTAL, 1)
    li, gi, hi = walk.branch_hessian_diagonal()
    assert rel_err(li, lw) < RTOL and grad_err(gi, gw) < RTOL and grad_err(hi, hw) < RTOL
    walk.close()
    gen.close()


@gpu
def test_hessian_tip_partials_not_01():
    """tip partials that are not 0/1 vectors: the walk declines, the resident route answers"""
    pb = branch_problem(4, 9, 200, 4, 5, tip_states=False)
    pb.tip_partials = pb.tip_partials * np.random.default_rng(1).uniform(0.5, 1.0, pb.tip_partials.shape)
    tlk = make(pb)
    lnl, grad, hess = tlk.branch_hessian_diagonal()
    assert tlk.last_kernels() != RAN_WALK
    full = O.evaluate(pb)
    assert rel_err(lnl, full["lnl"]) < RTOL and grad_err(grad, full["grad"]) < RTOL
    assert grad_err(hess, oracle_hessian(pb)) < RTOL
    tlk.close()


@gpu
@pytest.mark.parametrize("S,C", [(4, 4), (20, 2)], ids=["nuc4", "aa20"])
def test_hessian_under_forced_rescaling(S, C):
    pb = branch_problem(S, 10, 120, C, 17 + S)
    tlk = make(pb)
    tlk.set_option(OPT_SCALING_THRESHOLD_EXP, 2)  # 1e-2: scaling actually fires on this small tree
    tlk.use_rescaling(True)
    lnl, grad, hess = tlk.branch_hessian_diagonal()
    full = O.evaluate(pb)
    assert rel_err(lnl, full["lnl"]) < RTOL
    assert grad_err(grad, full["grad"]) < RTOL
    assert grad_err(hess, oracle_hessian(pb)) < RTOL
    tlk.close()


@gpu
def test_hessian_deep_caterpillar_switches_rescaling_on():
    """a tree whose site likelihoods underflow unscaled: the call switches rescaling on, recomputes, and returns finite values equal to
    the single-branch path's"""
    T, P = 640, 64
    topo = syn.caterpillar_topology(T)
    m = models.gtr([0.05, 0.3, 0.1, 0.15, 0.3, 0.1], [0.1, 0.2, 0.3, 0.4])
    rates, props = models.discrete_gamma(0.5, 4)
    bl = np.random.default_rng(2).uniform(0.5, 1.0, topo.nnodes)
    bl[topo.root] = 0.0
    pb = O.Problem(left=topo.left, right=topo.right, parent=topo.parent, root=topo.root, nstate=4,
                   tip_states=syn.random_patterns(T, P, 4, 0.25, 3), weights=np.ones(P), freqs=m.freqs, rates=rates, props=props, bl=bl,
                   evec=m.evec, eval=m.eval, ivec=m.ivec)
    pb.unrooted = False
    tlk = make(pb)
    assert not tlk.rescaling()
    lnl, grad, hess = tlk.branch_hessian_diagonal()
    assert tlk.rescaling()
    assert np.isfinite(lnl) and lnl / P < -745  # the average site likelihood is below the smallest double
    assert np.all(np.isfinite(grad)) and np.all(np.isfinite(hess))
    nodes = [n for n in range(0, topo.nnodes, 37) if n != topo.root] + [topo.left[topo.root], topo.right[topo.root]]
    for n in nodes:
        l1, d1, d2 = tlk.calculate_branch(n, [bl[n]])
        assert rel_err(l1[0], lnl) < RTOL
        assert abs(d1[0] - grad[n]) <= RTOL * max(abs(d1[0]), 1e-6 * np.abs(grad).max())
        assert abs(d2[0] - hess[n]) <= RTOL * max(abs(d2[0]), 1e-6 * np.abs(hess).max())
    tlk.close()


@gpu
@pytest.mark.parametrize("S,C", [(4, 4), (20, 2)], ids=["nuc4", "aa20"])
def test_hessian_central_differences_of_gradient(S, C):
    pb = branch_problem(S, 12, 400, C, 23 + S)
    tlk = make(pb)
    lnl, grad, hess = tlk.branch_hessian_diagonal()
    fd = np.zeros(pb.nnodes)
    for n in range(pb.nnodes):
        if n == pb.root:
            continue
        h = 1e-5 * pb.bl[n]
        g = []
        for s in (1.0, -1.0):
            tlk.set_branch_length(n, pb.bl[n] + s * h)
            g.append(tlk.gradient()[n])
        tlk.set_branch_length(n, pb.bl[n])
        fd[n] = (g[0] - g[1]) / (2 * h)
    assert grad_err(hess, fd) < 1e-6
    tlk.close()


@gpu
@pytest.mark.parametrize("S", [4, 20])
def test_hessian_conventions(S):
    pb = synthetic_problem(S, 10, 150, 4, 60 + S)  # unrooted: the root's right child has length 0 and a zero entry
    assert pb.unrooted
    tlk = make(pb)
    lnl, grad, hess = tlk.branch_hessian_diagonal()
    r = pb.right[pb.root]
    assert hess[pb.root] == 0.0 and hess[r] == 0.0 and grad[pb.root] == 0.0 and grad[r] == 0.0
    full = O.evaluate(pb)
    assert grad_err(grad, full["grad"]) < RTOL
    want = oracle_hessian(pb)
    want[r] = 0.0
    assert grad_err(hess, want) < RTOL
    # the cached lnL is the returned one: calculate() launches nothing
    before = tlk.launch_count()
    assert tlk.calculate() == lnl
    assert tlk.launch_count() == before
    # run-to-run bit-identical
    l2, g2, h2 = tlk.branch_hessian_diagonal()
    assert l2 == lnl and np.array_equal(g2, grad) and np.array_equal(h2, hess)
    # the gradient buffer the object owns still answers on its own
    assert grad_err(tlk.gradient(), full["grad"]) < RTOL
    tlk.close()


@gpu
def test_hessian_explicit_matrices_refused():
    pb = synthetic_problem(4, 6, 50, 2, 3)
    tlk = make(pb)
    tlk.gradient()
    Pm, dPm = tlk.get_matrices()
    tlk.set_matrices(Pm, dPm)
    with pytest.raises(phb.PhysherB200Error, match=r"^\[-4\]"):
        tlk.branch_hessian_diagonal()
    tlk.close()
