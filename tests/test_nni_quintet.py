"""Quintet scores of the NNI neighbourhood in one call (phb_tlk_nni_quintet_scores): lnL, gradient and Hessian in the five branches of
each exchanged tree -- the central branch c = v, keep and x at v's end, y and the fourth branch o at the far end (kind R: p's own branch,
none when p is the root; kind C: keep_w's branch) -- from resident partials and without a topology change.

Reference values: the oracle (oracle.branch_derivatives) on the exchanged Problem with the five lengths set; the off-diagonal Hessian
entries from central differences of the oracle's first derivatives, and exactly from spr_tripod_scores on the exchanged tree where the
three branches of a pair meet at one node.  On trees that underflow unscaled, the device's own set_topology + calculate_branch.
Tolerance: RTOL with the grad_err convention of tests/util.py.
"""
import numpy as np
import pytest

import physher_b200 as phb
from oracle import oracle as O
from physher_b200 import models, synthetic as syn
from physher_b200.treelikelihood import OPT_SCALING_THRESHOLD_EXP, OPT_UNROOTED, _dp, _ip
from tests.test_branch_hessian import branch_problem, make
from tests.test_nni import IDS, SHAPES, exchange
from tests.test_score_geometry import GRID_Y, big_trees, largest_s, launches, refusal, sample  # noqa: F401 (big_trees: fixture)
from tests.util import RTOL, grad_err, rel_err

pytestmark = pytest.mark.gpu

IU = np.triu_indices(5)  # the order of out[6:]: cc ck cx cy co kk kx ky ko xx xy xo yy yo oo


def sibling(pb, n):
    p = int(pb.parent[n])
    return int(pb.right[p] if pb.left[p] == n else pb.left[p])


def five(pb, x, y):
    """nodes (c, k, x, y, o) of move (x, y); o is None when p is the root (kind R)"""
    x, y = int(x), int(y)
    v = int(pb.parent[y])
    p = int(pb.parent[v])
    if int(pb.parent[x]) == p:  # kind R
        o = None if p == int(pb.root) else p
    else:  # kind C: the child of w that stays
        o = sibling(pb, x)
    return [v, sibling(pb, y), x, y, o]


def defaults(pb, moves):
    return np.array([[pb.bl[n] if n is not None else 0.0 for n in five(pb, x, y)] for x, y in moves])


def quintet_tree(pb, x, y, t5):
    q = exchange(pb, int(x), int(y))
    for n, t in zip(five(pb, x, y), t5):
        if n is not None:
            q.bl[n] = t
    return q


def raw(res):
    """(lnl[n], grad[n, 5], hess[n, 5, 5]) back to the C layout [n][21]"""
    lnl, g, h = res
    return np.column_stack([lnl, g, h[:, IU[0], IU[1]]])


def diag_col(a):
    return 6 + int(np.flatnonzero((IU[0] == a) & (IU[1] == a))[0])


def pair_col(a, b):
    a, b = min(a, b), max(a, b)
    return 6 + int(np.flatnonzero((IU[0] == a) & (IU[1] == b))[0])


def grad_of(pb, x, y, t5, a):
    q = quintet_tree(pb, x, y, t5)
    return O.branch_derivatives(q, five(pb, x, y)[a], [t5[a]])[0][1]


def mixed(pb, x, y, t5, a, b, rel=1e-5):
    """d g_a / d t_b by a central difference of the oracle's g_a"""
    h = rel * max(t5[b], 1e-3)
    g = []
    for sgn in (1, -1):
        t = np.array(t5, dtype=np.float64)
        t[b] += sgn * h
        g.append(grad_of(pb, x, y, t, a))
    return (g[0] - g[1]) / (2 * h)


def oracle_quintet(pb, moves, t5, nmixed=0):
    """[n][21]: lnL, the five first derivatives and the five diagonal entries from the oracle; the mixed entries of the first nmixed moves
    from central differences (the mean of both orders, which must agree), NaN for the rest; every entry of an absent o is 0"""
    out = np.full((len(moves), 21), np.nan)
    for k, (x, y) in enumerate(moves):
        nodes = five(pb, x, y)
        q = quintet_tree(pb, x, y, t5[k])
        for a, n in enumerate(nodes):
            if n is None:
                out[k, 1 + a] = 0.0
                out[k, [pair_col(a, b) for b in range(5)]] = 0.0
                continue
            d = O.branch_derivatives(q, n, [t5[k][a]])[0]
            out[k, 0], out[k, 1 + a], out[k, diag_col(a)] = d
        if k >= nmixed:
            continue
        for a in range(5):
            for b in range(a + 1, 5):
                if nodes[a] is None or nodes[b] is None:
                    continue
                ab, ba = mixed(pb, x, y, t5[k], a, b), mixed(pb, x, y, t5[k], b, a)
                assert abs(ab - ba) <= 1e-5 * max(abs(out[k, diag_col(a)]), abs(out[k, diag_col(b)]), 1e-6)  # both orders agree
                out[k, pair_col(a, b)] = 0.5 * (ab + ba)
    return out


def check(got, want, mixed_tol=1e-5):
    assert np.max(np.abs(got[:, 0] - want[:, 0]) / np.abs(want[:, 0])) < RTOL
    for col in range(1, 21):
        known = ~np.isnan(want[:, col])
        if not known.any():
            continue
        is_mixed = col >= 6 and IU[0][col - 6] != IU[1][col - 6]
        assert grad_err(got[known, col], want[known, col]) < (mixed_tol if is_mixed else RTOL), col


def random_five(pb, moves, seed):
    return defaults(pb, moves) * np.random.default_rng(seed).uniform(0.3, 3.0, (len(moves), 5))


# ---------------------------------------------------------------------------------------------------------------------------------
# 1. every move against the oracle
# ---------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("S,C,tip_states,T,P", SHAPES, ids=IDS)
def test_every_move_against_oracle(S, C, tip_states, T, P):
    pb = branch_problem(S, T, P, C, 70 + S + T, tip_states)
    tlk = make(pb)
    for unrooted in (True, False):
        tlk.set_option(OPT_UNROOTED, int(unrooted))
        moves = tlk.nni_moves()
        if len(moves) == 0:
            continue
        for t5, nmixed in ((None, 2), (random_five(pb, moves, 7 + S), 2)):
            got = raw(tlk.nni_quintet_scores(moves, t5))
            want = oracle_quintet(pb, moves, defaults(pb, moves) if t5 is None else t5, nmixed)
            check(got, want)
    tlk.close()


# ---------------------------------------------------------------------------------------------------------------------------------
# 2. exact mixed entries from the tripod scores of the exchanged tree
# ---------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("S,C", [(4, 4), (20, 2)], ids=["nuc4", "aa20"])
def test_mixed_entries_from_tripod_scores(S, C):
    pb = branch_problem(S, 12, 200, C, 300 + S)
    tlk = make(pb)
    tlk.set_option(OPT_UNROOTED, 0)
    moves = tlk.nni_moves()
    r1, r2 = int(pb.left[pb.root]), int(pb.right[pb.root])
    if pb.left[r1] >= 0 and pb.left[r2] >= 0:  # kind C moves too
        moves = np.concatenate([moves, np.array([[pb.left[r1], pb.left[r2]], [pb.left[r2], pb.right[r1]]], np.int32)])
    got = raw(tlk.nni_quintet_scores(moves))
    other = tlk.clone()
    compared = 0
    for k, (x, y) in enumerate(moves):
        c, kp, xx, yy, o = five(pb, x, y)
        q = exchange(pb, int(x), int(y))
        other.set_topology(q.left, q.right, q.root)
        size = np.max(np.abs(got[k, 6:]))
        # s = keep, b = x: (up, down, pend) = (c, x, k)
        _, _, h = other.spr_tripod_scores(kp, [xx], [[pb.bl[c], pb.bl[xx], pb.bl[kp]]])
        for (a, b), (i, j) in (((0, 2), (0, 1)), ((0, 1), (0, 2)), ((2, 1), (1, 2))):
            assert abs(got[k, pair_col(a, b)] - h[0, i, j]) <= 1e-10 * size
        if o is not None:  # y hangs from u = p (kind R) or w (kind C), neither the root
            u = int(q.parent[yy])
            b = int(q.right[u] if q.left[u] == yy else q.left[u])
            if b == c:  # kind R, s = y, b = v: (up, down, pend) = (o, c, y)
                _, _, h = other.spr_tripod_scores(yy, [c], [[pb.bl[o], pb.bl[c], pb.bl[yy]]])
                pairs = (((4, 0), (0, 1)), ((4, 3), (0, 2)), ((0, 3), (1, 2)))
            else:  # kind C, s = y, b = o: (up, down, pend) = (w, o, y), of which (o, y) is a quintet pair
                _, _, h = other.spr_tripod_scores(yy, [o], [[pb.bl[u], pb.bl[o], pb.bl[yy]]])
                pairs = (((4, 3), (1, 2)),)
            for (a, b), (i, j) in pairs:
                assert abs(got[k, pair_col(a, b)] - h[0, i, j]) <= 1e-10 * size
        compared += 1
    assert compared == len(moves)
    other.close()
    tlk.close()


# ---------------------------------------------------------------------------------------------------------------------------------
# 3. reduction to nni_scores, 4. directional differences
# ---------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("S,C", [(4, 4), (20, 2), (61, 1), (5, 3)], ids=["nuc4", "aa20", "codon61", "generic5"])
def test_reduces_to_nni_scores(S, C):
    pb = branch_problem(S, 10, 150, C, 320 + S)
    tlk = make(pb)
    moves = tlk.nni_moves()
    lnl0, ref = tlk.nni_scores(moves)
    lnl, g, h = tlk.nni_quintet_scores(moves)
    assert np.max(np.abs(lnl - ref[:, 0]) / np.abs(ref[:, 0])) < 1e-12
    assert grad_err(g[:, 0], ref[:, 1]) < 1e-10
    assert grad_err(h[:, 0, 0], ref[:, 2]) < 1e-10
    tlk.close()


@pytest.mark.parametrize("S,C", [(4, 4), (20, 2)], ids=["nuc4", "aa20"])
def test_directional_differences(S, C):
    pb = branch_problem(S, 10, 300, C, 340 + S)
    tlk = make(pb)
    moves = tlk.nni_moves()
    t5 = random_five(pb, moves, 11)
    d = t5 * np.random.default_rng(S).uniform(-1.0, 1.0, t5.shape)
    lnl, g, H = tlk.nni_quintet_scores(moves, t5)
    h1 = 1e-5
    up, _, _ = tlk.nni_quintet_scores(moves, t5 + h1 * d)
    dn, _, _ = tlk.nni_quintet_scores(moves, t5 - h1 * d)
    assert grad_err((up - dn) / (2 * h1), np.einsum("ka,ka->k", g, d)) < 1e-6

    def second(h):
        up, _, _ = tlk.nni_quintet_scores(moves, t5 + h * d)
        dn, _, _ = tlk.nni_quintet_scores(moves, t5 - h * d)
        return (up - 2 * lnl + dn) / h ** 2

    h2 = 1e-2  # Richardson on the second difference: the h^2 term cancels
    assert grad_err((4 * second(h2 / 2) - second(h2)) / 3, np.einsum("ka,kab,kb->k", d, H, d), floor=1e-3) < 1e-5
    tlk.close()


# ---------------------------------------------------------------------------------------------------------------------------------
# 5. edge cases
# ---------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("S,C", [(4, 4), (20, 2), (5, 1)], ids=["nuc4", "aa20", "generic5"])
def test_cross_root_and_root_moves(S, C):
    """kind C moves (valid in rooted mode too) against the oracle; rooted moves with p the root have every o entry exactly 0"""
    pb = branch_problem(S, 12, 300, C, 81)
    r1, r2 = int(pb.left[pb.root]), int(pb.right[pb.root])
    if pb.left[r1] < 0 or pb.left[r2] < 0:  # both root children internal
        pb = branch_problem(S, 12, 300, C, 82)
        r1, r2 = int(pb.left[pb.root]), int(pb.right[pb.root])
    assert pb.left[r1] >= 0 and pb.left[r2] >= 0
    tlk = make(pb)
    tlk.set_option(OPT_UNROOTED, 0)
    cross = np.array([[pb.left[r1], pb.left[r2]], [pb.right[r1], pb.right[r2]], [pb.left[r2], pb.left[r1]], [pb.right[r2], pb.right[r1]]],
                     np.int32)
    t5 = random_five(pb, cross, 13)
    check(raw(tlk.nni_quintet_scores(cross, t5)), oracle_quintet(pb, cross, t5, 2))
    moves = tlk.nni_moves()
    at_root = np.array([k for k, (x, y) in enumerate(moves) if five(pb, x, y)[4] is None])
    assert len(at_root) == 4
    got = raw(tlk.nni_quintet_scores(moves[at_root]))
    assert np.all(got[:, [5] + [pair_col(a, 4) for a in range(5)]] == 0.0)
    check(got, oracle_quintet(pb, moves[at_root], defaults(pb, moves[at_root]), 1))
    # the order of the list does not change a move's numbers
    _, g, h = tlk.nni_quintet_scores(moves)
    perm = np.random.default_rng(3).permutation(len(moves))
    _, g2, h2 = tlk.nni_quintet_scores(moves[perm])
    assert np.array_equal(g2, g[perm]) and np.array_equal(h2, h[perm])
    tlk.close()


# ---------------------------------------------------------------------------------------------------------------------------------
# 6. rescaling and the object's state
# ---------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("S,C", [(4, 4), (20, 2)], ids=["nuc4", "aa20"])
def test_forced_rescaling(S, C):
    pb = branch_problem(S, 10, 120, C, 360 + S)
    tlk = make(pb)
    tlk.set_option(OPT_SCALING_THRESHOLD_EXP, 2)  # 1e-2: scaling fires on this small tree
    tlk.use_rescaling(True)
    moves = tlk.nni_moves()
    t5 = random_five(pb, moves, 17)
    check(raw(tlk.nni_quintet_scores(moves, t5)), oracle_quintet(pb, moves, t5))
    tlk.close()


def device_reference(other, pb, x, y, t5):
    """lnL and the five (g, H) diagonal pairs of the exchanged tree from set_topology + calculate_branch"""
    q = quintet_tree(pb, x, y, t5)
    other.set_topology(q.left, q.right, q.root)
    other.set_branch_lengths(q.bl)
    out = []
    for n, t in zip(five(pb, x, y), t5):
        lnl, d1, d2 = other.calculate_branch(n, [t])
        out.append((lnl[0], d1[0], d2[0]))
    return out


def test_deep_caterpillar_switches_rescaling_on():
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
    moves = moves[[k for k, (x, y) in enumerate(moves) if five(pb, x, y)[4] is not None]]
    t5 = random_five(pb, moves, 19)
    lnl, g, h = tlk.nni_quintet_scores(moves, t5)
    assert tlk.rescaling()
    assert np.all(np.isfinite(lnl)) and np.all(np.isfinite(g)) and np.all(np.isfinite(h))
    other = make(pb)
    other.use_rescaling(True)
    for k in list(range(0, len(moves), 157)) + [len(moves) - 1]:
        ref = device_reference(other, pb, moves[k][0], moves[k][1], t5[k])
        for a, (l, d1, d2) in enumerate(ref):
            assert rel_err(lnl[k], l) < RTOL
            assert abs(g[k, a] - d1) <= RTOL * max(abs(d1), 1e-6)
            assert abs(h[k, a, a] - d2) <= RTOL * max(abs(d2), 1e-6)
    other.close()
    tlk.close()


def test_neighbour_underflow_switches_rescaling_on():
    """the current tree is finite unscaled, one neighbour's site likelihood is 0: rescaling comes on, the call scores once more, the
    other moves still match the oracle and the impossible one is -inf"""
    T, P = 8, 200
    topo = syn.caterpillar_topology(T)
    H = np.array([[1, 1, 1, 1], [1, -1, 1, -1], [1, 1, -1, -1], [1, -1, -1, 1]], dtype=np.float64)
    evec, ivec, evals = H, H / 4, np.array([0.0, -4 / 3, -4 / 3, -4 / 3])  # P(0) is the identity exactly
    rates, props = models.discrete_gamma(0.5, 4)
    bl = np.random.default_rng(5).uniform(0.05, 0.3, topo.nnodes)
    bl[topo.root] = 0.0
    cherry = next(n for n in range(T, topo.nnodes) if topo.left[n] < T and topo.right[n] < T)
    t1, t2 = int(topo.left[cherry]), int(topo.right[cherry])
    p = int(topo.parent[cherry])
    t3 = int(topo.left[p] if topo.right[p] == cherry else topo.right[p])
    assert t3 < T
    bl[t2] = bl[t3] = 0.0  # after move (t3, t1) the zero-length tips t2, t3 share a parent: L = 0 wherever their states differ
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
    got = raw(tlk.nni_quintet_scores(moves))
    assert tlk.rescaling()
    assert got[zero[0], 0] == -np.inf
    rest = np.array([k for k in range(len(moves)) if k != zero[0]])
    check(got[rest], oracle_quintet(pb, moves[rest], defaults(pb, moves[rest])))
    tlk.close()


@pytest.mark.parametrize("S", [4, 20, 61])
def test_object_state_after_the_call(S):
    pb = branch_problem(S, 11, 200, 2 if S == 61 else 4, 380 + S)
    tlk = make(pb)
    full = O.evaluate(pb)
    moves = tlk.nni_moves()
    lnl0, _ = tlk.nni_scores(moves)  # PHB_OPT_INCREMENTAL on, as the quintet call leaves it
    assert rel_err(lnl0, full["lnl"]) < RTOL

    def state():
        g = tlk.gradient().copy()
        h = tlk.branch_hessian_diagonal()
        _, o = tlk.nni_scores(moves)
        return tlk.calculate(), g, h[1].copy(), h[2].copy(), o

    before = state()
    got = tlk.nni_quintet_scores(moves, random_five(pb, moves, 23))
    n = tlk.launch_count()
    assert tlk.calculate() == before[0]  # the cached lnL, unchanged
    assert tlk.launch_count() == n
    after = state()
    for x, y in zip(before, after):
        assert np.array_equal(x, y)
    again = tlk.nni_quintet_scores(moves, random_five(pb, moves, 23))
    assert all(np.array_equal(x, y) for x, y in zip(got, again))
    tlk.close()


# ---------------------------------------------------------------------------------------------------------------------------------
# 7. launch geometry and refusals
# ---------------------------------------------------------------------------------------------------------------------------------
# the any-S kernel keeps 12 S-vectors of 32 patterns up to 16 states, 16 up to 32 and 8 past that (at most 92 KiB at 120 states); "max2"
# is the largest state count the node-at-a-time kernels accept, read from the device
@pytest.mark.parametrize("S", [2, 5, 26, 27, 61, "max2"])
def test_state_counts(S):
    S = largest_s(2) if S == "max2" else S
    pb = branch_problem(S, 7, 40, 2, 400 + S)
    tlk = make(pb)
    tlk.set_option(OPT_UNROOTED, 0)
    moves = tlk.nni_moves()
    t5 = random_five(pb, moves, 29)
    check(raw(tlk.nni_quintet_scores(moves, t5)), oracle_quintet(pb, moves, t5, 1))
    tlk.close()


@pytest.mark.parametrize("S", [4, 5])
def test_moves_past_one_launch(big_trees, S):
    pb = big_trees(S, 33000)
    tlk = make(pb)
    moves = tlk.nni_moves()
    assert len(moves) > GRID_Y + 1
    tlk.nni_quintet_scores(moves[:2])
    n_two, _ = launches(tlk, tlk.nni_quintet_scores, moves[:2])
    n_all, res = launches(tlk, tlk.nni_quintet_scores, moves)
    print(f"NNI quintet, {S} states: {len(moves)} moves, {n_all} launches, 2 moves: {n_two}")
    assert n_all == n_two + 1
    got = raw(res)
    k = sample(len(moves), 6, 4)
    check(got[k], oracle_quintet(pb, moves[k], defaults(pb, moves[k])))
    perm = np.random.default_rng(5).permutation(len(moves))
    assert np.array_equal(raw(tlk.nni_quintet_scores(moves[perm])), got[perm])
    tlk.close()


def test_refused_past_the_state_count_limit():
    S = largest_s(2) + 1
    pb = branch_problem(S, 5, 16, 1, 440)
    tlk = make(pb)
    moves = tlk.nni_moves()
    for _ in range(2):  # refused before any launch, the same way every time
        before = tlk.launch_count()
        with pytest.raises(phb.PhysherB200Error, match=refusal(S, 2)):
            tlk.nni_quintet_scores(moves)
        assert tlk.launch_count() == before
    tlk.close()


def test_refusals():
    pb = branch_problem(4, 9, 50, 2, 450)
    tlk = make(pb)
    moves = tlk.nni_moves()
    bad = moves.copy()
    bad[3] = [int(pb.root), int(bad[3][1])]
    with pytest.raises(phb.PhysherB200Error, match=r"^\[-1\].*move 3"):
        tlk.nni_quintet_scores(bad)
    y = int(moves[0][1])  # a move whose x is y's own parent
    with pytest.raises(phb.PhysherB200Error, match=r"^\[-1\].*move 0"):
        tlk.nni_quintet_scores(np.array([[pb.parent[y], y]]))
    with pytest.raises(phb.PhysherB200Error, match=r"^\[-1\]"):
        tlk.nni_quintet_scores(moves[:0])
    t5 = defaults(pb, moves[:2])
    for j in range(5):
        for v in (-0.1, np.nan):
            t = t5.copy()
            t[1, j] = v
            with pytest.raises(phb.PhysherB200Error, match=r"^\[-1\].*move 1"):
                tlk.nni_quintet_scores(moves[:2], t)
    one = np.ascontiguousarray(moves[:1], np.int32)
    out = np.zeros(21)
    assert tlk.lib.phb_tlk_nni_quintet_scores(tlk.h, 1, None, None, None, out.ctypes.data_as(_dp)) == -1
    assert tlk.lib.phb_tlk_nni_quintet_scores(tlk.h, 1, one.ctypes.data_as(_ip), None, None, None) == -1
    assert tlk.lib.phb_tlk_nni_quintet_scores(tlk.h, 0, one.ctypes.data_as(_ip), None, None, out.ctypes.data_as(_dp)) == -1
    # the object still works
    check(raw(tlk.nni_quintet_scores(moves)), oracle_quintet(pb, moves, defaults(pb, moves)))
    assert rel_err(tlk.calculate(), O.evaluate(pb, gradient=False)["lnl"]) < RTOL
    tlk.gradient()
    Pm, dPm = tlk.get_matrices()
    tlk.set_matrices(Pm, dPm)
    with pytest.raises(phb.PhysherB200Error, match=r"^\[-4\]"):
        tlk.nni_quintet_scores(moves)
    tlk.close()
