"""Scores of the NNI neighbourhood in one call (phb_tlk_nni_moves / phb_tlk_nni_scores): lnL, d lnL/dt_v and d2 lnL/dt_v2 of the tree
each nearest-neighbour interchange produces, from resident partials and without a topology change.

Reference values: the oracle (oracle.evaluate, oracle.branch_derivatives) on the exchanged Problem; on a tree that underflows
unscaled, the device's own set_topology + calculate.  Tolerance: RTOL with the grad_err convention of tests/util.py.
"""
import copy

import numpy as np
import pytest

import physher_b200 as phb
from oracle import oracle as O
from physher_b200 import models, synthetic as syn
from physher_b200.treelikelihood import OPT_SCALING_THRESHOLD_EXP, OPT_UNROOTED
from tests.test_branch_hessian import branch_problem, make
from tests.util import RTOL, grad_err, rel_err

pytestmark = pytest.mark.gpu


def exchange(pb, x, y):
    """the tree of move (x, y): x takes y's slot under v = parent[y], y takes x's slot under parent[x]; lengths stay with node ids"""
    left, right, parent = pb.left.copy(), pb.right.copy(), pb.parent.copy()
    v, u = int(parent[y]), int(parent[x])
    if left[v] == y:
        left[v] = x
    else:
        right[v] = x
    if left[u] == x:
        left[u] = y
    else:
        right[u] = y
    parent[x], parent[y] = v, u
    q = copy.copy(pb)
    q.left, q.right, q.parent = left, right, parent
    q.bl = pb.bl.copy()
    return q


def oracle_scores(pb, moves, t_central=None):
    out = np.zeros((len(moves), 3))
    for k, (x, y) in enumerate(moves):
        v = int(pb.parent[y])
        q = exchange(pb, int(x), int(y))
        t = pb.bl[v] if t_central is None else t_central[k]
        q.bl[v] = t
        out[k] = O.branch_derivatives(q, v, [t])[0]
    return out


def check(got, want):
    assert np.max(np.abs(got[:, 0] - want[:, 0]) / np.abs(want[:, 0])) < RTOL
    assert grad_err(got[:, 1], want[:, 1]) < RTOL
    assert grad_err(got[:, 2], want[:, 2]) < RTOL


def splits(left, right, root, T):
    """non-trivial splits of the unrooted tree, each as the side without tip 0"""
    below = {}

    def walk(n):
        if left[n] < 0:
            below[n] = frozenset([n])
        else:
            below[n] = walk(left[n]) | walk(right[n])
        return below[n]

    walk(root)
    tips = frozenset(range(T))
    out = set()
    for n, s in below.items():
        if n == root:
            continue
        side = s if 0 not in s else tips - s
        if 1 < len(side) < T - 1:
            out.add(side)
    return frozenset(out)


SHAPES = [  # S, C, tip_states, T, P
    (4, 4, True, 9, 301), (4, 1, False, 9, 301), (4, 8, True, 9, 301), (20, 4, True, 9, 301), (20, 2, False, 9, 301), (61, 1, True, 9, 301),
    (5, 3, True, 9, 301), (4, 4, True, 9, 1), (20, 4, True, 9, 1), (4, 4, True, 3, 301), (4, 4, True, 4, 301), (20, 1, True, 4, 77),
]
IDS = ["nuc4-g4", "nuc4-partials", "nuc4-c8", "aa20-g4", "aa20-partials", "codon61", "generic5", "nuc4-p1", "aa20-p1", "nuc4-t3",
       "nuc4-t4", "aa20-t4"]


@pytest.mark.parametrize("S,C,tip_states,T,P", SHAPES, ids=IDS)
def test_every_move_against_oracle(S, C, tip_states, T, P):
    pb = branch_problem(S, T, P, C, 70 + S + T, tip_states)
    tlk = make(pb)
    full = O.evaluate(pb)
    for unrooted in (True, False):
        tlk.set_option(OPT_UNROOTED, int(unrooted))
        moves = tlk.nni_moves()
        assert len(moves) == (2 * (T - 3) if unrooted else 2 * (T - 2))
        if len(moves) == 0:
            continue
        lnl, out = tlk.nni_scores()
        assert rel_err(lnl, full["lnl"]) < RTOL
        check(out, oracle_scores(pb, moves))
    tlk.close()


def test_explicit_lists_cross_root_moves_and_order():
    pb = branch_problem(4, 12, 400, 4, 81)
    r1, r2 = int(pb.left[pb.root]), int(pb.right[pb.root])
    if pb.left[r1] < 0 or pb.left[r2] < 0:  # both root children internal
        pb = branch_problem(4, 12, 400, 4, 82)
        r1, r2 = int(pb.left[pb.root]), int(pb.right[pb.root])
    assert pb.left[r1] >= 0 and pb.left[r2] >= 0
    tlk = make(pb)
    tlk.set_option(OPT_UNROOTED, 0)  # kind C moves are valid in rooted mode too
    cross = np.array([[pb.left[r1], pb.left[r2]], [pb.right[r1], pb.right[r2]], [pb.left[r2], pb.left[r1]], [pb.right[r2], pb.right[r1]]],
                     np.int32)
    moves = np.concatenate([cross, tlk.nni_moves()])
    _, out = tlk.nni_scores(moves)
    check(out, oracle_scores(pb, moves))
    perm = np.random.default_rng(3).permutation(len(moves))
    _, out2 = tlk.nni_scores(moves[perm])
    assert np.array_equal(out2, out[perm])  # each move is formed the same way in whichever group and slot it lands
    tlk.close()


@pytest.mark.parametrize("S,C", [(4, 4), (20, 2)], ids=["nuc4", "aa20"])
def test_candidate_lengths(S, C):
    pb = branch_problem(S, 10, 300, C, 90 + S)
    tlk = make(pb)
    moves = tlk.nni_moves()
    v = pb.parent[moves[:, 1]]
    tc = pb.bl[v] * np.random.default_rng(4).uniform(0.3, 3.0, len(moves))
    _, out = tlk.nni_scores(moves, tc)
    check(out, oracle_scores(pb, moves, tc))
    # central differences of lnL in t_central
    h = 1e-5 * tc
    _, up = tlk.nni_scores(moves, tc + h)
    _, dn = tlk.nni_scores(moves, tc - h)
    assert grad_err((up[:, 0] - dn[:, 0]) / (2 * h), out[:, 1]) < 1e-6
    assert grad_err((up[:, 1] - dn[:, 1]) / (2 * h), out[:, 2]) < 1e-6
    # a call that changes only t_central: the matrix table, the score kernel(s) and the sum
    before = tlk.launch_count()
    _, again = tlk.nni_scores(moves, tc)
    assert tlk.launch_count() - before == (3 if S == 4 else 4)
    assert np.array_equal(again, out)
    fresh = make(pb)
    _, f = fresh.nni_scores(moves, tc)
    assert np.array_equal(f, out)
    fresh.close()
    tlk.close()


@pytest.mark.parametrize("T", [2, 3, 4, 9, 30])
def test_enumeration(T):
    pb = branch_problem(4, T, 20, 1, 100 + T)
    tlk = make(pb)
    tlk.set_option(OPT_UNROOTED, 1)
    moves = tlk.nni_moves()
    assert len(moves) == max(0, 2 * (T - 3))
    base = splits(pb.left, pb.right, pb.root, T)
    seen = set()
    for x, y in moves:
        q = exchange(pb, int(x), int(y))
        s = splits(q.left, q.right, q.root, T)
        assert len(s - base) == 1 and len(base - s) == 1
        seen.add(s)
    assert len(seen) == len(moves)
    tlk.set_option(OPT_UNROOTED, 0)
    assert len(tlk.nni_moves()) == max(0, 2 * (T - 2))
    tlk.close()


@pytest.mark.parametrize("S,C", [(4, 4), (20, 2)], ids=["nuc4", "aa20"])
def test_forced_rescaling(S, C):
    pb = branch_problem(S, 10, 120, C, 110 + S)
    tlk = make(pb)
    tlk.set_option(OPT_SCALING_THRESHOLD_EXP, 2)  # 1e-2: scaling fires on this small tree
    tlk.use_rescaling(True)
    moves = tlk.nni_moves()
    lnl, out = tlk.nni_scores(moves)
    assert rel_err(lnl, O.evaluate(pb, gradient=False)["lnl"]) < RTOL
    check(out, oracle_scores(pb, moves))
    tlk.close()


def test_deep_caterpillar_switches_rescaling_on():
    """site likelihoods underflow unscaled: rescaling comes on, every score is finite and matches set_topology + calculate"""
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
    moves = tlk.nni_moves()
    lnl, out = tlk.nni_scores(moves)
    assert tlk.rescaling()
    assert np.isfinite(lnl) and lnl / P < -745
    assert np.all(np.isfinite(out))
    other = make(pb)
    other.use_rescaling(True)
    for k in list(range(0, len(moves), 97)) + [len(moves) - 1]:
        x, y = (int(a) for a in moves[k])
        q = exchange(pb, x, y)
        other.set_topology(q.left, q.right, q.root)
        assert rel_err(out[k, 0], other.calculate()) < RTOL
        _, d1, d2 = other.calculate_branch(int(pb.parent[y]), [bl[pb.parent[y]]])
        assert abs(out[k, 1] - d1[0]) <= RTOL * max(abs(d1[0]), 1e-6)
        assert abs(out[k, 2] - d2[0]) <= RTOL * max(abs(d2[0]), 1e-6)
    other.close()
    tlk.close()


def test_neighbour_underflow_switches_rescaling_on():
    """the current tree is finite unscaled, one neighbour's site likelihood is 0: rescaling comes on, the call scores once more, the
    other moves still match the oracle and the impossible one is -inf"""
    T, P = 8, 200
    topo = syn.caterpillar_topology(T)
    # JC69 with the Hadamard eigenvectors: every term of P(0) is a power of two, so P(0) is the identity exactly and a zero-length
    # branch passes a tip's 0/1 vector through without rounding
    H = np.array([[1, 1, 1, 1], [1, -1, 1, -1], [1, 1, -1, -1], [1, -1, -1, 1]], dtype=np.float64)
    evec, ivec, evals = H, H / 4, np.array([0.0, -4 / 3, -4 / 3, -4 / 3])
    rates, props = models.discrete_gamma(0.5, 4)
    bl = np.random.default_rng(5).uniform(0.05, 0.3, topo.nnodes)
    bl[topo.root] = 0.0
    cherry = next(n for n in range(T, topo.nnodes) if topo.left[n] < T and topo.right[n] < T)
    t1, t2 = int(topo.left[cherry]), int(topo.right[cherry])
    p = int(topo.parent[cherry])
    t3 = int(topo.left[p] if topo.right[p] == cherry else topo.right[p])
    assert t3 < T
    bl[t2] = bl[t3] = 0.0  # after move (t3, t1) the two zero-length tips t2, t3 share a parent: L = 0 wherever their states differ
    st = syn.random_patterns(T, P, 4, 0.25, 6)
    assert np.any((st[t2] != st[t3]) & (st[t2] < 4) & (st[t3] < 4))
    pb = O.Problem(left=topo.left, right=topo.right, parent=topo.parent, root=topo.root, nstate=4, tip_states=st, weights=np.ones(P),
                   freqs=np.full(4, 0.25), rates=rates, props=props, bl=bl, evec=evec, eval=evals, ivec=ivec)
    pb.unrooted = False
    tlk = make(pb)
    assert np.isfinite(tlk.calculate()) and not tlk.rescaling()
    moves = tlk.nni_moves()
    zero = [k for k, (x, y) in enumerate(moves) if x == t3 and y == t1]
    assert len(zero) == 1
    lnl, out = tlk.nni_scores(moves)
    assert tlk.rescaling()
    assert rel_err(lnl, O.evaluate(pb, gradient=False)["lnl"]) < RTOL
    assert out[zero[0], 0] == -np.inf
    rest = np.array([k for k in range(len(moves)) if k != zero[0]])
    check(out[rest], oracle_scores(pb, moves[rest]))
    tlk.close()


def test_any_state_route_in_several_chunks(monkeypatch):
    """the any-S route with its operand scratch capped at three moves: the same values as one chunk, two launches per chunk"""
    pb = branch_problem(20, 12, 150, 2, 140)
    tlk = make(pb)
    moves = tlk.nni_moves()
    lnl, one = tlk.nni_scores(moves)
    monkeypatch.setenv("PHB_NNI_CHUNK_MOVES", "3")
    before = tlk.launch_count()
    l2, chunked = tlk.nni_scores(moves)
    assert tlk.launch_count() - before == 2 + 2 * ((len(moves) + 2) // 3)
    assert l2 == lnl and np.array_equal(chunked, one)
    check(chunked, oracle_scores(pb, moves))
    tlk.close()


@pytest.mark.parametrize("S", [4, 20])
def test_object_state_after_the_call(S):
    pb = branch_problem(S, 11, 200, 4, 120 + S)
    tlk = make(pb)
    full = O.evaluate(pb)
    lnl, out = tlk.nni_scores()
    assert rel_err(lnl, full["lnl"]) < RTOL
    # the cached lnL is the returned one: calculate() launches nothing
    before = tlk.launch_count()
    assert tlk.calculate() == lnl
    assert tlk.launch_count() == before
    # topology and branch lengths unchanged: the object still evaluates the original tree
    assert grad_err(tlk.gradient(), full["grad"]) < RTOL
    tlk.update_all_nodes()
    assert rel_err(tlk.calculate(), full["lnl"]) < RTOL
    # run-to-run bit-identical
    l2, out2 = tlk.nni_scores()
    assert l2 == lnl and np.array_equal(out2, out)
    tlk.close()


def test_refusals():
    pb = branch_problem(4, 8, 50, 2, 130)
    tlk = make(pb)
    moves = tlk.nni_moves()
    bad = moves.copy()
    bad[3] = [int(pb.root), int(bad[3][1])]
    with pytest.raises(phb.PhysherB200Error, match=r"^\[-1\].*move 3"):
        tlk.nni_scores(bad)
    with pytest.raises(phb.PhysherB200Error, match=r"^\[-1\]"):
        tlk.nni_scores(moves[:0])
    with pytest.raises(phb.PhysherB200Error, match=r"^\[-1\].*move 0"):
        tlk.nni_scores(moves[:1], [-0.1])
    y = int(moves[0][1])  # a move whose x is y's own parent
    with pytest.raises(phb.PhysherB200Error, match=r"^\[-1\]"):
        tlk.nni_scores(np.array([[pb.parent[y], y]]))
    # the object still works
    lnl, out = tlk.nni_scores(moves)
    check(out, oracle_scores(pb, moves))
    assert rel_err(lnl, O.evaluate(pb, gradient=False)["lnl"]) < RTOL
    tlk.gradient()
    Pm, dPm = tlk.get_matrices()
    tlk.set_matrices(Pm, dPm)
    with pytest.raises(phb.PhysherB200Error, match=r"^\[-4\]"):
        tlk.nni_scores(moves)
    tlk.close()
