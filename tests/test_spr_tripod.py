"""Tripod scores of every regraft of a pruned subtree in one call (phb_tlk_spr_tripod_scores): lnL, gradient and Hessian in the three
branches that meet at the regraft point -- node p's (t_up), the target e's (t_down) and s's (t_pend) -- of the tree each subtree
prune-and-regraft move produces, with b's branch joined in the pruned tree, from one pass over the pruned tree's resident partials.

Reference values: the oracle (oracle.evaluate, oracle.branch_derivatives) on the regrafted Problem with bl[p] = t_up, bl[e] = t_down,
bl[s] = t_pend and bl[b] = l_b (e != b); the off-diagonal Hessian entries from central differences of the oracle's first derivatives.
On trees that underflow unscaled, the device's own set_topology + calculate_branch.  Tolerance: RTOL with the grad_err convention of
tests/util.py.
"""
import numpy as np
import pytest

import physher_b200 as phb
from oracle import oracle as O
from physher_b200 import models, synthetic as syn
from physher_b200.treelikelihood import OPT_SCALING_THRESHOLD_EXP, OPT_UNROOTED, _dp, _ip
from tests.test_branch_hessian import branch_problem, make
from tests.test_nni import IDS, SHAPES
from tests.test_score_geometry import GRID_Y, big_trees, largest_s, launches, refusal, sample  # noqa: F401 (big_trees: fixture)
from tests.test_spr import _scaled, depth, ntips, prunable, prune_choices, regraft, sibling
from tests.util import RTOL, grad_err, rel_err

pytestmark = pytest.mark.gpu

PAIRS = [(0, 1), (0, 2), (1, 2)]  # (up, down), (up, pend), (down, pend): out columns 7, 8, 9


def raw(res):
    """(lnl[n], grad[n, 3], hess[n, 3, 3]) back to the C layout [n][10]"""
    lnl, g, h = res
    return np.column_stack([lnl, g, h[:, 0, 0], h[:, 1, 1], h[:, 2, 2], h[:, 0, 1], h[:, 0, 2], h[:, 1, 2]])


def defaults(pb, s, targets, join=None):
    """the call's defaults: l_b = t_b + t_p (or join), t_up = t_down = l_e / 2, t_pend = t_s"""
    p, b = int(pb.parent[s]), sibling(pb, s)
    lb = pb.bl[b] + pb.bl[p] if join is None else join
    half = np.array([(lb if e == b else pb.bl[e]) / 2 for e in targets])
    return lb, np.column_stack([half, half, np.full(len(targets), pb.bl[s])])


def tripod_tree(pb, s, e, tri, lb):
    q = regraft(pb, s, int(e))
    q.bl[sibling(pb, s)] = lb
    p = int(pb.parent[s])
    q.bl[p], q.bl[int(e)], q.bl[s] = tri
    return q


def nodes_of(pb, s, e):
    return [int(pb.parent[s]), int(e), int(s)]


def oracle_tripod(pb, s, targets, tri, lb, nmixed=0):
    """[n][10]; the mixed entries of the first nmixed targets from central differences of the oracle's first derivatives (the mean of
    both orders, which must agree with each other), NaN for the rest"""
    out = np.full((len(targets), 10), np.nan)
    for k, e in enumerate(targets):
        q = tripod_tree(pb, s, e, tri[k], lb)
        nodes = nodes_of(pb, s, e)
        for a in range(3):
            d = O.branch_derivatives(q, nodes[a], [tri[k][a]])[0]
            out[k, 0], out[k, 1 + a], out[k, 4 + a] = d[0], d[1], d[2]
        if k >= nmixed:
            continue
        for col, (a, b) in zip((7, 8, 9), PAIRS):
            ab, ba = mixed(pb, s, e, tri[k], lb, a, b), mixed(pb, s, e, tri[k], lb, b, a)
            assert abs(ab - ba) <= 1e-5 * max(abs(out[k, 4 + a]), abs(out[k, 4 + b]), 1e-6)  # both orders agree
            out[k, col] = 0.5 * (ab + ba)
    return out


def mixed(pb, s, e, tri, lb, a, b, rel=1e-5):
    """d g_a / d t_b by a central difference of the oracle's g_a"""
    h = rel * max(tri[b], 1e-3)
    g = []
    for sgn in (1, -1):
        t = np.array(tri, dtype=np.float64)
        t[b] += sgn * h
        q = tripod_tree(pb, s, e, t, lb)
        g.append(O.branch_derivatives(q, nodes_of(pb, s, e)[a], [t[a]])[0][1])
    return (g[0] - g[1]) / (2 * h)


def check(got, want, mixed_tol=1e-5):
    """lnL, gradient and Hessian diagonal within RTOL; the mixed entries where want has them, within what the difference step allows"""
    assert np.max(np.abs(got[:, 0] - want[:, 0]) / np.abs(want[:, 0])) < RTOL
    for col in range(1, 7):
        assert grad_err(got[:, col], want[:, col]) < RTOL, col
    rows = ~np.isnan(want[:, 7])
    if rows.any():
        scale = max(np.abs(want[:, 4:7]).max(), 1e-300)  # the Hessian's own size
        assert np.max(np.abs(got[rows, 7:] - want[rows, 7:])) / scale < mixed_tol


def random_tripod(pb, s, targets, seed):
    _, d = defaults(pb, s, targets)
    return d * np.random.default_rng(seed).uniform(0.3, 3.0, d.shape)


# ---------------------------------------------------------------------------------------------------------------------------------
# 1. every target against the oracle
# ---------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("S,C,tip_states,T,P", SHAPES, ids=IDS)
def test_every_target_against_oracle(S, C, tip_states, T, P):
    pb = branch_problem(S, T, P, C, 370 + S + T, tip_states)
    tlk = make(pb)
    for unrooted in (True, False):
        tlk.set_option(OPT_UNROOTED, int(unrooted))
        for s in prune_choices(pb):
            targets = tlk.spr_targets(s)
            if len(targets) == 0:
                continue
            b, p = sibling(pb, s), int(pb.parent[s])
            # default tripod and join; random tripod lengths with an explicit join
            join = (pb.bl[b] + pb.bl[p]) * np.random.default_rng(s).uniform(0.5, 1.5)
            for tri, tj in ((None, None), (random_tripod(pb, s, targets, 10 + s), join)):
                got = raw(tlk.spr_tripod_scores(s, targets, tri, tj))
                lb, dflt = defaults(pb, s, targets, tj)
                nmixed = 3 if (tri is not None and not unrooted) else 0
                want = oracle_tripod(pb, s, targets, dflt if tri is None else tri, lb, nmixed)
                check(got, want)
    tlk.close()


# ---------------------------------------------------------------------------------------------------------------------------------
# 2. / 3. the existing calls: spr_scores at the current lengths, and target b as the current tree
# ---------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("S,C", [(4, 4), (20, 2), (61, 1), (5, 3)], ids=["nuc4", "aa20", "codon61", "generic5"])
def test_reduces_to_spr_scores(S, C):
    pb = branch_problem(S, 10, 200, C, 380 + S)
    tlk = make(pb)
    for s in prune_choices(pb):
        targets = tlk.spr_targets(s)
        p, b = int(pb.parent[s]), sibling(pb, s)
        tri = np.column_stack([np.full(len(targets), pb.bl[p]), pb.bl[targets], np.full(len(targets), pb.bl[s])])
        got = raw(tlk.spr_tripod_scores(s, targets, tri, pb.bl[b]))
        _, spr = tlk.spr_scores(s, targets)
        assert np.max(np.abs(got[:, 0] - spr[:, 0]) / np.abs(spr[:, 0])) < RTOL
        assert grad_err(got[:, 3], spr[:, 1]) < RTOL
        assert grad_err(got[:, 6], spr[:, 2]) < RTOL
    tlk.close()


@pytest.mark.parametrize("S,C", [(4, 4), (20, 2), (61, 1)], ids=["nuc4", "aa20", "codon61"])
def test_target_b_is_the_current_tree(S, C):
    pb = branch_problem(S, 12, 200, C, 390 + S)
    ref = make(pb)
    ref.set_option(OPT_UNROOTED, 0)
    lnl0 = ref.calculate()
    g0 = ref.gradient().copy()
    _, _, h0 = ref.branch_hessian_diagonal()
    tlk = make(pb)
    for s in prunable(pb):
        p, b = int(pb.parent[s]), sibling(pb, s)
        got = raw(tlk.spr_tripod_scores(s, [b], [[pb.bl[p], pb.bl[b], pb.bl[s]]]))[0]
        assert rel_err(got[0], lnl0) < RTOL
        for a, n in enumerate((p, b, s)):
            assert abs(got[1 + a] - g0[n]) <= RTOL * max(abs(g0[n]), 1e-6), (s, a)
            assert abs(got[4 + a] - h0[n]) <= RTOL * max(abs(h0[n]), 1e-6), (s, a)
    tlk.close()
    ref.close()


# ---------------------------------------------------------------------------------------------------------------------------------
# 4. directional derivatives of the device's own lnL
# ---------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("S,C", [(4, 4), (20, 2)], ids=["nuc4", "aa20"])
def test_directional_differences(S, C):
    pb = branch_problem(S, 10, 300, C, 400 + S)
    tlk = make(pb)
    rng = np.random.default_rng(S)
    for s in prune_choices(pb):
        targets = tlk.spr_targets(s)
        tri = random_tripod(pb, s, targets, 20 + s)
        d = tri * rng.uniform(-1.0, 1.0, tri.shape)
        lnl, g, H = tlk.spr_tripod_scores(s, targets, tri)
        h1 = 1e-5
        up, _, _ = tlk.spr_tripod_scores(s, targets, tri + h1 * d)
        dn, _, _ = tlk.spr_tripod_scores(s, targets, tri - h1 * d)
        assert grad_err((up - dn) / (2 * h1), np.einsum("ka,ka->k", g, d)) < 1e-6

        def second(h):
            up, _, _ = tlk.spr_tripod_scores(s, targets, tri + h * d)
            dn, _, _ = tlk.spr_tripod_scores(s, targets, tri - h * d)
            return (up - 2 * lnl + dn) / h ** 2

        # Richardson on the second difference: the h^2 term cancels.  The rounding of lnL (~1e-12 of |lnL| ~ 7e3) over h^2 is ~3e-8,
        # so entries are compared on at least 1e-3 of the largest |dT H d|
        h2 = 1e-2
        assert grad_err((4 * second(h2 / 2) - second(h2)) / 3, np.einsum("ka,kab,kb->k", d, H, d), floor=1e-3) < 1e-5
    tlk.close()


# ---------------------------------------------------------------------------------------------------------------------------------
# 5. rescaling
# ---------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("S,C", [(4, 4), (20, 2)], ids=["nuc4", "aa20"])
def test_forced_rescaling(S, C):
    pb = branch_problem(S, 10, 120, C, 410 + S)
    tlk = make(pb)
    tlk.set_option(OPT_SCALING_THRESHOLD_EXP, 2)  # 1e-2: scaling fires on this small tree
    tlk.use_rescaling(True)
    for s in prune_choices(pb):
        targets = tlk.spr_targets(s)
        tri = random_tripod(pb, s, targets, 30 + s)
        got = raw(tlk.spr_tripod_scores(s, targets, tri))
        lb, _ = defaults(pb, s, targets)
        check(got, oracle_tripod(pb, s, targets, tri, lb, 2))
    tlk.close()


def device_reference(other, pb, s, e, tri, lb):
    """lnL and the three (d1, d2) of the regrafted tree from a device object with rescaling on: set_topology + calculate_branch"""
    q = tripod_tree(pb, s, e, tri, lb)
    other.set_topology(q.left, q.right, q.root)
    other.set_branch_lengths(q.bl)
    out = np.zeros(7)
    out[0] = other.calculate()
    for a, n in enumerate(nodes_of(pb, s, e)):
        _, d1, d2 = other.calculate_branch(n, [tri[a]])
        out[1 + a], out[4 + a] = d1[0], d2[0]
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
    s = max(prunable(pb), key=lambda n: (depth(pb, n), -int(pb.left[n] >= 0)))
    targets = tlk.spr_targets(s)
    got = raw(tlk.spr_tripod_scores(s, targets))
    assert tlk.rescaling()
    assert np.all(np.isfinite(got))
    lb, tri = defaults(pb, s, targets)
    other = make(pb)
    other.use_rescaling(True)
    for k in list(range(0, len(targets), 97)) + [len(targets) - 1]:
        want = device_reference(other, pb, s, targets[k], tri[k], lb)
        assert rel_err(got[k, 0], want[0]) < RTOL
        for col in range(1, 7):
            assert abs(got[k, col] - want[col]) <= RTOL * max(abs(want[col]), 1e-6), (k, col)
    other.close()
    tlk.close()


def jc_hadamard():
    H = np.array([[1, 1, 1, 1], [1, -1, 1, -1], [1, 1, -1, -1], [1, -1, -1, 1]], dtype=np.float64)
    return H, H / 4, np.array([0.0, -4 / 3, -4 / 3, -4 / 3])  # P(0) is the identity exactly


def test_target_underflow_switches_rescaling_on():
    """one regrafted tree's site likelihood is exactly 0 (s and e next to each other at zero length with different states): rescaling
    comes on, that target's lnL is -inf and every other target matches the oracle"""
    T, P = 8, 200
    topo = syn.caterpillar_topology(T)
    evec, ivec, evals = jc_hadamard()
    rates, props = models.discrete_gamma(0.5, 4)
    bl = np.random.default_rng(5).uniform(0.05, 0.3, topo.nnodes)
    bl[topo.root] = 0.0
    st = syn.random_patterns(T, P, 4, 0.25, 6)
    s, e = next((a, c) for a in range(T) for c in range(T) if a != c and topo.parent[a] != topo.root and topo.parent[a] != topo.parent[c]
                and np.any((st[a] != st[c]) & (st[a] < 4) & (st[c] < 4)))
    pb = O.Problem(left=topo.left, right=topo.right, parent=topo.parent, root=topo.root, nstate=4, tip_states=st, weights=np.ones(P),
                   freqs=np.full(4, 0.25), rates=rates, props=props, bl=bl, evec=evec, eval=evals, ivec=ivec)
    pb.unrooted = False
    tlk = make(pb)
    assert np.isfinite(tlk.calculate()) and not tlk.rescaling()
    targets = tlk.spr_targets(s)
    lb, tri = defaults(pb, s, targets)
    zero = int(np.flatnonzero(targets == e)[0])
    tri[zero, 1:] = 0.0
    got = raw(tlk.spr_tripod_scores(s, targets, tri))
    assert tlk.rescaling()
    assert got[zero, 0] == -np.inf
    rest = np.array([k for k in range(len(targets)) if k != zero])
    check(got[rest], oracle_tripod(pb, s, targets[rest], tri[rest], lb))
    tlk.close()


def test_target_that_underflows_unscaled_is_scored_after_rescaling():
    """a regrafted tree whose site likelihood underflows to 0 unscaled but is not 0: rescaling comes on, the call scores once more and
    that target gets its finite score"""
    T = 520  # a caterpillar whose site likelihood sits near the bottom of the double range (lnL ~ -722), above it
    topo = syn.caterpillar_topology(T)
    evec, ivec, evals = jc_hadamard()
    st = np.random.default_rng(9).integers(0, 4, (T, 1)).astype(np.uint8)
    bl = np.ones(topo.nnodes)
    bl[topo.root] = 0.0
    pb = O.Problem(left=topo.left, right=topo.right, parent=topo.parent, root=topo.root, nstate=4, tip_states=st, weights=np.ones(1),
                   freqs=np.full(4, 0.25), rates=np.ones(1), props=np.ones(1), bl=bl, evec=evec, eval=evals, ivec=ivec)
    pb.unrooted = False
    s = next(a for a in prunable(pb) if a < T)
    e = next(c for c in range(T - 1, -1, -1) if st[c, 0] != st[s, 0] and topo.parent[c] != topo.parent[s])
    bl[e] = 0.0
    pb.bl = bl
    p, b = int(pb.parent[s]), sibling(pb, s)
    tiny = 1e-16
    tri_e = [bl[p], 0.0, tiny]  # the regrafted tree of spr_scores' test, b kept at t_b
    q = tripod_tree(pb, s, e, tri_e, bl[b])
    assert np.isfinite(O.evaluate(pb, gradient=False)["lnl"])
    assert O.evaluate(q, gradient=False)["lnl"] == -np.inf
    want = O.evaluate(_scaled(q), gradient=False)["lnl"]
    assert np.isfinite(want)
    tlk = make(pb)
    assert np.isfinite(tlk.calculate()) and not tlk.rescaling()
    targets = tlk.spr_targets(s)
    k = int(np.flatnonzero(targets == e)[0])
    tri = np.column_stack([np.full(len(targets), bl[p]), bl[targets], np.full(len(targets), bl[s])])
    tri[k] = tri_e
    got = raw(tlk.spr_tripod_scores(s, targets, tri, bl[b]))
    assert tlk.rescaling()
    assert np.all(np.isfinite(got))
    assert rel_err(got[k, 0], want) < RTOL
    other = make(pb)
    other.use_rescaling(True)
    for j in (k, 0, len(targets) - 1):
        ref = device_reference(other, pb, s, targets[j], tri[j], bl[b])
        assert rel_err(got[j, 0], ref[0]) < RTOL
        for col in range(1, 7):
            assert abs(got[j, col] - ref[col]) <= RTOL * max(abs(ref[col]), 1e-6), (j, col)
    other.close()
    tlk.close()


# ---------------------------------------------------------------------------------------------------------------------------------
# 6. the object after the call
# ---------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("S", [4, 20, 61])
def test_object_state_after_the_call(S):
    """the joined length does not leak: calculate, gradient, the Hessian diagonal and spr_scores return the bits they returned before,
    for every kind of s (b's matrix rebuilt at l_b and back, g the root or not); repeats and reorderings are bit-identical"""
    pb = branch_problem(S, 11, 200, 2 if S == 61 else 4, 420 + S)
    tlk = make(pb)
    full = O.evaluate(pb)
    picks = prune_choices(pb)
    probe = picks[-1]
    lnl0, _ = tlk.spr_scores(probe)  # PHB_OPT_INCREMENTAL on, as the tripod call leaves it
    assert rel_err(lnl0, full["lnl"]) < RTOL

    def state():
        g = tlk.gradient().copy()
        h = tlk.branch_hessian_diagonal()
        _, o = tlk.spr_scores(probe)
        return g, h[1].copy(), h[2].copy(), o

    before = state()
    for s in picks:
        targets = tlk.spr_targets(s)
        got = tlk.spr_tripod_scores(s, targets)
        n = tlk.launch_count()
        assert tlk.calculate() == lnl0
        assert tlk.launch_count() == n
        after = state()
        for x, y in zip(before, after):
            assert np.array_equal(x, y), s
        again = tlk.spr_tripod_scores(s, targets)
        assert all(np.array_equal(x, y) for x, y in zip(got, again))
        perm = np.random.default_rng(s).permutation(len(targets))
        shuffled = tlk.spr_tripod_scores(s, targets[perm])
        assert all(np.array_equal(x, y[perm]) for x, y in zip(shuffled, got))
    assert tlk.calculate() == lnl0
    tlk.update_all_nodes()
    assert rel_err(tlk.calculate(), full["lnl"]) < RTOL
    tlk.close()


# ---------------------------------------------------------------------------------------------------------------------------------
# 7. launch geometry and refusals
# ---------------------------------------------------------------------------------------------------------------------------------
# the any-S kernel stages its nine matrices whole up to 26 states (9 x 26^2 x 8 = 48,672 bytes) and a chunk of rows past it (27 states:
# 25 rows, 2 chunks; 61: 11 rows, 6 chunks); 20 and 61 run on the tensor-core pruned pass with host exponentials (61); "max2" is the
# largest state count the pruned pass's node-at-a-time kernels accept, read from the device
@pytest.mark.parametrize("S", [2, 5, 26, 27, 61, "max2"])
def test_state_counts(S):
    S = largest_s(2) if S == "max2" else S
    pb = branch_problem(S, 7, 40, 2, 430 + S)
    tlk = make(pb)
    for s in prune_choices(pb)[:2]:
        targets = tlk.spr_targets(s)
        tri = random_tripod(pb, s, targets, 40 + s)
        got = raw(tlk.spr_tripod_scores(s, targets, tri))
        lb, _ = defaults(pb, s, targets)
        check(got, oracle_tripod(pb, s, targets, tri, lb, 1))
    tlk.close()


@pytest.mark.parametrize("S", [4, 5])
def test_targets_past_one_launch(big_trees, S):
    pb = big_trees(S, 33000)
    tlk = make(pb)
    s = next(n for n in prunable(pb) if pb.left[n] < 0)
    targets = tlk.spr_targets(s)
    assert len(targets) > GRID_Y + 1
    tlk.spr_tripod_scores(s, targets[:2])
    n_two, _ = launches(tlk, tlk.spr_tripod_scores, s, targets[:2])
    n_all, res = launches(tlk, tlk.spr_tripod_scores, s, targets)
    print(f"SPR tripod of tip {s}: {len(targets)} targets, {n_all} launches, 2 targets: {n_two}")
    assert n_all == n_two + 1
    got = raw(res)
    k = sample(len(targets), 6, 4)
    lb, tri = defaults(pb, s, targets)
    want = np.zeros((len(k), 7))
    for j, kk in enumerate(k):
        q = tripod_tree(pb, s, targets[kk], tri[kk], lb)
        for a, n in enumerate(nodes_of(pb, s, targets[kk])):
            d = O.branch_derivatives(q, n, [tri[kk][a]])[0]
            want[j, 0], want[j, 1 + a], want[j, 4 + a] = d
    assert np.max(np.abs(got[k, 0] - want[:, 0]) / np.abs(want[:, 0])) < RTOL
    for col in range(1, 7):
        assert grad_err(got[k, col], want[:, col]) < RTOL, col
    perm = np.random.default_rng(5).permutation(len(targets))
    assert np.array_equal(raw(tlk.spr_tripod_scores(s, targets[perm])), got[perm])
    tlk.close()


def test_refused_past_the_state_count_limit():
    S = largest_s(2) + 1
    pb = branch_problem(S, 5, 16, 1, 440)
    tlk = make(pb)
    s = prune_choices(pb)[0]
    for _ in range(2):  # refused before any launch, the same way every time
        before = tlk.launch_count()
        with pytest.raises(phb.PhysherB200Error, match=refusal(S, 2)):
            tlk.spr_tripod_scores(s, tlk.spr_targets(s))
        assert tlk.launch_count() == before
    with pytest.raises(phb.PhysherB200Error, match=refusal(S, 2)):
        tlk.calculate()
    tlk.close()


def test_refusals():
    pb = branch_problem(4, 9, 50, 2, 450)
    tlk = make(pb)
    r = int(pb.root)
    for bad in (r, int(pb.left[r]), int(pb.right[r]), -1, pb.nnodes):
        with pytest.raises(phb.PhysherB200Error, match=r"^\[-1\]"):
            tlk.spr_tripod_scores(bad, [0])
    s = min((n for n in prunable(pb) if pb.left[n] >= 0), key=lambda n: ntips(pb, n))
    targets = tlk.spr_targets(s)
    assert len(targets) >= 4
    for e in (int(pb.parent[s]), r, s, int(pb.left[s]), -1, pb.nnodes):
        bad = targets.copy()
        bad[3] = e
        with pytest.raises(phb.PhysherB200Error, match=r"^\[-1\].*target 3"):
            tlk.spr_tripod_scores(s, bad)
    with pytest.raises(phb.PhysherB200Error, match=r"^\[-1\]"):
        tlk.spr_tripod_scores(s, targets[:0])
    tri = np.ones((2, 3)) * 0.1
    for j in range(3):
        for v in (-0.1, np.nan):
            t = tri.copy()
            t[1, j] = v
            with pytest.raises(phb.PhysherB200Error, match=r"^\[-1\].*target 1"):
                tlk.spr_tripod_scores(s, targets[:2], t)
    for v in (-0.1, np.nan):
        with pytest.raises(phb.PhysherB200Error, match=r"^\[-1\].*joined"):
            tlk.spr_tripod_scores(s, targets[:2], tri, v)
    one = np.array(targets[:1], np.int32)
    assert tlk.lib.phb_tlk_spr_tripod_scores(tlk.h, s, 1, None, None, None, None, None) == -1
    assert tlk.lib.phb_tlk_spr_tripod_scores(tlk.h, s, 1, one.ctypes.data_as(_ip), None, None, None, None) == -1
    out = np.zeros(10)
    assert tlk.lib.phb_tlk_spr_tripod_scores(tlk.h, s, 0, one.ctypes.data_as(_ip), None, None, None, out.ctypes.data_as(_dp)) == -1
    # the object still works
    got = raw(tlk.spr_tripod_scores(s, targets))
    lb, dflt = defaults(pb, s, targets)
    check(got, oracle_tripod(pb, s, targets, dflt, lb))
    assert rel_err(tlk.calculate(), O.evaluate(pb, gradient=False)["lnl"]) < RTOL
    tlk.gradient()
    Pm, dPm = tlk.get_matrices()
    tlk.set_matrices(Pm, dPm)
    with pytest.raises(phb.PhysherB200Error, match=r"^\[-4\]"):
        tlk.spr_tripod_scores(s, targets)
    tlk.close()
