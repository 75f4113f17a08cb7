"""Scores of every regraft of a pruned subtree in one call (phb_tlk_spr_targets / phb_tlk_spr_scores): lnL, d lnL/dt_s and d2 lnL/dt_s2
of the tree each subtree prune-and-regraft move produces, from one pass over the pruned tree's resident partials and without a
topology change.

Reference values: the oracle (oracle.evaluate, oracle.branch_derivatives) on the regrafted Problem; on a tree that underflows unscaled,
the device's own set_topology + calculate.  Tolerance: RTOL with the grad_err convention of tests/util.py.
"""
import copy

import numpy as np
import pytest

import physher_b200 as phb
from oracle import oracle as O
from physher_b200 import models, synthetic as syn
from physher_b200.treelikelihood import OPT_SCALING_THRESHOLD_EXP, OPT_UNROOTED, _ip
from tests.test_branch_hessian import branch_problem, make
from tests.test_nni import IDS, SHAPES, check, splits
from tests.util import RTOL, grad_err, rel_err

pytestmark = pytest.mark.gpu


def sibling(pb, n):
    u = pb.parent[n]
    return int(pb.right[u] if pb.left[u] == n else pb.left[u])


def regraft(pb, s, e):
    """the tree of the move (s, e): p = parent[s] and the subtree of s pruned (the sibling b of s takes p's slot under g = parent[p]),
    then p takes e's slot under e's parent in the pruned tree and e the slot of p that is not s's; lengths stay with node ids"""
    left, right, parent = pb.left.copy(), pb.right.copy(), pb.parent.copy()
    p = int(parent[s])
    g, b = int(parent[p]), sibling(pb, s)
    if left[g] == p:
        left[g] = b
    else:
        right[g] = b
    parent[b] = g
    h = int(parent[e])
    if left[h] == e:
        left[h] = p
    else:
        right[h] = p
    parent[p] = h
    if left[p] == s:
        right[p] = e
    else:
        left[p] = e
    parent[e] = p
    q = copy.copy(pb)
    q.left, q.right, q.parent = left, right, parent
    q.bl = pb.bl.copy()
    return q


def oracle_scores(pb, s, targets, t_pendant=None):
    out = np.zeros((len(targets), 3))
    for k, e in enumerate(targets):
        q = regraft(pb, s, int(e))
        t = pb.bl[s] if t_pendant is None else t_pendant[k]
        q.bl[s] = t
        out[k] = O.branch_derivatives(q, s, [t])[0]
    return out


def subtree(pb, s):
    out, stack = [], [s]
    while stack:
        x = stack.pop()
        out.append(x)
        if pb.left[x] >= 0:
            stack += [int(pb.left[x]), int(pb.right[x])]
    return out


def ntips(pb, s):
    return sum(1 for x in subtree(pb, s) if pb.left[x] < 0)


def depth(pb, n):
    d = 0
    while n != pb.root:
        n, d = int(pb.parent[n]), d + 1
    return d


def prunable(pb):
    return [n for n in range(pb.nnodes) if n != pb.root and pb.parent[n] != pb.root]


def prune_choices(pb):
    """a tip, an internal node, a node whose grandparent is the root and the deepest node, each where the tree has one"""
    cand = prunable(pb)
    picks = [next((n for n in cand if pb.left[n] < 0), None), next((n for n in cand if pb.left[n] >= 0), None),
             next((n for n in cand if pb.parent[pb.parent[n]] == pb.root), None), max(cand, key=lambda n: depth(pb, n))]
    return sorted({int(n) for n in picks if n is not None})


@pytest.mark.parametrize("S,C,tip_states,T,P", SHAPES, ids=IDS)
def test_every_target_against_oracle(S, C, tip_states, T, P):
    pb = branch_problem(S, T, P, C, 170 + S + T, tip_states)
    tlk = make(pb)
    full = O.evaluate(pb, gradient=False)
    for unrooted in (True, False):
        tlk.set_option(OPT_UNROOTED, int(unrooted))
        for s in prune_choices(pb):
            targets = tlk.spr_targets(s)
            k = ntips(pb, s)
            assert len(targets) == (2 * (T - k) - 4 if unrooted else 2 * (T - k) - 3)
            if len(targets) == 0:
                continue
            lnl, out = tlk.spr_scores(s)
            assert rel_err(lnl, full["lnl"]) < RTOL
            check(out, oracle_scores(pb, s, targets))
    tlk.close()


@pytest.mark.parametrize("T", [3, 4, 9, 30])
def test_enumeration(T):
    pb = branch_problem(4, T, 20, 1, 200 + T)
    tlk = make(pb)
    base = splits(pb.left, pb.right, pb.root, T)
    for s in prunable(pb):
        k, b = ntips(pb, s), sibling(pb, s)
        tlk.set_option(OPT_UNROOTED, 1)
        targets = tlk.spr_targets(s)
        assert len(targets) == 2 * (T - k) - 4
        seen = set()
        for e in targets:
            q = regraft(pb, s, int(e))
            sp = splits(q.left, q.right, q.root, T)
            assert sp != base
            seen.add(sp)
        assert len(seen) == len(targets)
        tlk.set_option(OPT_UNROOTED, 0)
        targets = tlk.spr_targets(s)
        assert len(targets) == 2 * (T - k) - 3
        assert b not in targets
        inside = set(subtree(pb, s)) | {int(pb.parent[s]), int(pb.root)}
        assert not inside & {int(e) for e in targets}
    tlk.close()


@pytest.mark.parametrize("S,C", [(4, 4), (20, 2)], ids=["nuc4", "aa20"])
def test_consistency_with_existing_calls(S, C):
    """target b is the current tree: lnL, gradient and Hessian diagonal entry of branch s; target q is the NNI move (q, b)"""
    pb = branch_problem(S, 12, 300, C, 210 + S)
    ref = make(pb)
    lnl0 = ref.calculate()
    g0 = ref.gradient().copy()
    _, _, h0 = ref.branch_hessian_diagonal()
    tlk = make(pb)
    for s in prunable(pb):
        b, q = sibling(pb, s), sibling(pb, int(pb.parent[s]))
        lnl, out = tlk.spr_scores(s, [b, q])
        assert rel_err(lnl, lnl0) < RTOL
        assert rel_err(out[0, 0], lnl0) < RTOL
        assert abs(out[0, 1] - g0[s]) <= RTOL * max(abs(g0[s]), 1e-6)
        assert abs(out[0, 2] - h0[s]) <= RTOL * max(abs(h0[s]), 1e-6)
        _, nni = ref.nni_scores(np.array([[q, b]], np.int32))
        assert rel_err(out[1, 0], nni[0, 0]) < RTOL
    tlk.close()
    ref.close()


@pytest.mark.parametrize("S,C", [(4, 4), (20, 2)], ids=["nuc4", "aa20"])
def test_candidate_pendant_lengths(S, C):
    pb = branch_problem(S, 10, 300, C, 220 + S)
    tlk = make(pb)
    for s in prune_choices(pb):
        targets = tlk.spr_targets(s)
        tp = pb.bl[s] * np.random.default_rng(s).uniform(0.3, 3.0, len(targets))
        _, out = tlk.spr_scores(s, targets, tp)
        check(out, oracle_scores(pb, s, targets, tp))
        h = 1e-5 * tp
        _, up = tlk.spr_scores(s, targets, tp + h)
        _, dn = tlk.spr_scores(s, targets, tp - h)
        assert grad_err((up[:, 0] - dn[:, 0]) / (2 * h), out[:, 1]) < 1e-6
        assert grad_err((up[:, 1] - dn[:, 1]) / (2 * h), out[:, 2]) < 1e-6
    tlk.close()


@pytest.mark.parametrize("S,C", [(4, 4), (20, 2)], ids=["nuc4", "aa20"])
def test_forced_rescaling(S, C):
    pb = branch_problem(S, 10, 120, C, 230 + S)
    tlk = make(pb)
    tlk.set_option(OPT_SCALING_THRESHOLD_EXP, 2)  # 1e-2: scaling fires on this small tree
    tlk.use_rescaling(True)
    want = O.evaluate(pb, gradient=False)["lnl"]
    for s in prune_choices(pb):
        targets = tlk.spr_targets(s)
        lnl, out = tlk.spr_scores(s, targets)
        assert rel_err(lnl, want) < RTOL
        check(out, oracle_scores(pb, s, targets))
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
    s = max(prunable(pb), key=lambda n: (depth(pb, n), -int(pb.left[n] >= 0)))  # a tip at the bottom of the caterpillar
    targets = tlk.spr_targets(s)
    lnl, out = tlk.spr_scores(s, targets)
    assert tlk.rescaling()
    assert np.isfinite(lnl) and lnl / P < -745
    assert np.all(np.isfinite(out))
    other = make(pb)
    other.use_rescaling(True)
    for k in list(range(0, len(targets), 97)) + [len(targets) - 1]:
        q = regraft(pb, s, int(targets[k]))
        other.set_topology(q.left, q.right, q.root)
        assert rel_err(out[k, 0], other.calculate()) < RTOL
        _, d1, d2 = other.calculate_branch(s, [bl[s]])
        assert abs(out[k, 1] - d1[0]) <= RTOL * max(abs(d1[0]), 1e-6)
        assert abs(out[k, 2] - d2[0]) <= RTOL * max(abs(d2[0]), 1e-6)
    other.close()
    tlk.close()


def test_target_underflow_switches_rescaling_on():
    """the current tree is finite unscaled, one regrafted tree's site likelihood is 0: rescaling comes on, the call scores once more,
    the other targets still match the oracle and the impossible one is -inf"""
    T, P = 8, 200
    topo = syn.caterpillar_topology(T)
    # JC69 with the Hadamard eigenvectors: P(0) is the identity exactly (see tests/test_nni.py)
    H = np.array([[1, 1, 1, 1], [1, -1, 1, -1], [1, 1, -1, -1], [1, -1, -1, 1]], dtype=np.float64)
    evec, ivec, evals = H, H / 4, np.array([0.0, -4 / 3, -4 / 3, -4 / 3])
    rates, props = models.discrete_gamma(0.5, 4)
    bl = np.random.default_rng(5).uniform(0.05, 0.3, topo.nnodes)
    bl[topo.root] = 0.0
    st = syn.random_patterns(T, P, 4, 0.25, 6)
    probe = O.Problem(left=topo.left, right=topo.right, parent=topo.parent, root=topo.root, nstate=4, tip_states=st, weights=np.ones(P),
                      freqs=np.full(4, 0.25), rates=rates, props=props, bl=bl, evec=evec, eval=evals, ivec=ivec)
    # two tips that are not siblings, the first prunable: regrafted next to each other at zero length, L = 0 where their states differ
    s, e = next((a, c) for a in range(T) for c in range(T) if a != c and topo.parent[a] != topo.root and topo.parent[a] != topo.parent[c]
                and np.any((st[a] != st[c]) & (st[a] < 4) & (st[c] < 4)))
    bl[s] = bl[e] = 0.0
    pb = probe
    pb.bl = bl
    pb.unrooted = False
    tlk = make(pb)
    assert np.isfinite(tlk.calculate()) and not tlk.rescaling()
    targets = tlk.spr_targets(s)
    zero = [k for k, x in enumerate(targets) if x == e]
    assert len(zero) == 1
    lnl, out = tlk.spr_scores(s, targets)
    assert tlk.rescaling()
    assert rel_err(lnl, O.evaluate(pb, gradient=False)["lnl"]) < RTOL
    assert out[zero[0], 0] == -np.inf
    rest = np.array([k for k in range(len(targets)) if k != zero[0]])
    check(out[rest], oracle_scores(pb, s, targets[rest]))
    tlk.close()


def test_target_that_underflows_unscaled_is_scored_after_rescaling():
    """the current tree is finite unscaled, one regrafted tree's site likelihood underflows to 0 unscaled but is not 0: rescaling comes
    on, the call scores once more and that target gets its finite score"""
    T = 520  # a caterpillar whose site likelihood sits near the bottom of the double range (lnL ~ -722), above it
    topo = syn.caterpillar_topology(T)
    # JC69 with the Hadamard eigenvectors (see tests/test_nni.py): P(0) is the identity exactly
    H = np.array([[1, 1, 1, 1], [1, -1, 1, -1], [1, 1, -1, -1], [1, -1, -1, 1]], dtype=np.float64)
    st = np.random.default_rng(9).integers(0, 4, (T, 1)).astype(np.uint8)
    bl = np.ones(topo.nnodes)
    bl[topo.root] = 0.0
    pb = O.Problem(left=topo.left, right=topo.right, parent=topo.parent, root=topo.root, nstate=4, tip_states=st, weights=np.ones(1),
                   freqs=np.full(4, 0.25), rates=np.ones(1), props=np.ones(1), bl=bl, evec=H, eval=np.array([0.0, -4 / 3, -4 / 3, -4 / 3]),
                   ivec=H / 4)
    pb.unrooted = False
    # s next to a zero-length tip e of another state, at a pendant length of 1e-16: a factor ~3e-17 takes the site likelihood below
    # the smallest double
    s = next(a for a in prunable(pb) if a < T)
    e = next(c for c in range(T - 1, -1, -1) if st[c, 0] != st[s, 0] and topo.parent[c] != topo.parent[s])
    bl[e] = 0.0
    pb.bl = bl
    tiny = 1e-16
    q = regraft(pb, s, e)
    q.bl[s] = tiny
    assert np.isfinite(O.evaluate(pb, gradient=False)["lnl"])
    assert O.evaluate(q, gradient=False)["lnl"] == -np.inf
    want = O.evaluate(_scaled(q), gradient=False)["lnl"]
    assert np.isfinite(want)
    tlk = make(pb)
    assert np.isfinite(tlk.calculate()) and not tlk.rescaling()
    targets = tlk.spr_targets(s)
    k = int(np.flatnonzero(targets == e)[0])
    tp = np.full(len(targets), bl[s])
    tp[k] = tiny
    lnl, out = tlk.spr_scores(s, targets, tp)
    assert tlk.rescaling()
    assert rel_err(lnl, O.evaluate(_scaled(pb), gradient=False)["lnl"]) < RTOL
    assert np.all(np.isfinite(out))
    assert rel_err(out[k, 0], want) < RTOL
    other = make(pb)
    other.use_rescaling(True)
    for j in (k, 0, len(targets) - 1):
        r = regraft(pb, s, int(targets[j]))
        other.set_topology(r.left, r.right, r.root)
        lj, d1, d2 = other.calculate_branch(s, [tp[j]])
        assert rel_err(out[j, 0], lj[0]) < RTOL
        assert abs(out[j, 1] - d1[0]) <= RTOL * max(abs(d1[0]), 1e-6)
        assert abs(out[j, 2] - d2[0]) <= RTOL * max(abs(d2[0]), 1e-6)
    other.close()
    tlk.close()


def _scaled(pb):
    q = copy.copy(pb)
    q.scale = True
    return q


@pytest.mark.parametrize("S", [4, 20])
def test_object_state_after_the_call(S):
    pb = branch_problem(S, 11, 200, 4, 240 + S)
    tlk = make(pb)
    full = O.evaluate(pb)
    s1, s2 = prune_choices(pb)[:2]
    lnl, out = tlk.spr_scores(s1)
    assert rel_err(lnl, full["lnl"]) < RTOL
    # the cached lnL is the returned one, bit for bit
    before = tlk.launch_count()
    assert tlk.calculate() == lnl
    assert tlk.launch_count() == before
    # the object still evaluates the original tree: the same answers as a fresh object
    fresh = make(pb)
    assert grad_err(tlk.gradient(), fresh.gradient()) < 1e-12
    _, nni = tlk.nni_scores()
    _, nni_f = fresh.nni_scores()
    assert grad_err(nni[:, 0], nni_f[:, 0]) < 1e-12 and grad_err(nni[:, 1:], nni_f[:, 1:]) < 1e-12
    _, o2 = tlk.spr_scores(s2)
    _, o2_f = fresh.spr_scores(s2)
    assert grad_err(o2[:, 0], o2_f[:, 0]) < 1e-12 and grad_err(o2[:, 1:], o2_f[:, 1:]) < 1e-12
    check(o2, oracle_scores(pb, s2, tlk.spr_targets(s2)))
    fresh.close()
    # run-to-run bit-identical, and independent of the order of the list
    targets = tlk.spr_targets(s1)
    l2, out2 = tlk.spr_scores(s1, targets)
    assert l2 == lnl and np.array_equal(out2, out)
    perm = np.random.default_rng(7).permutation(len(targets))
    _, out3 = tlk.spr_scores(s1, targets[perm])
    assert np.array_equal(out3, out[perm])
    assert tlk.calculate() == lnl
    tlk.update_all_nodes()
    assert rel_err(tlk.calculate(), full["lnl"]) < RTOL
    tlk.close()


def test_launch_count_does_not_grow_with_targets():
    """a repeat call launches the same kernels for 2 targets or all of them; past 65,535 targets one more score launch per grid.y slab"""
    pb = branch_problem(4, 12, 64, 2, 250)
    tlk = make(pb)
    s = prune_choices(pb)[0]
    targets = tlk.spr_targets(s)
    tlk.spr_scores(s, targets)

    def launches(tg):
        before = tlk.launch_count()
        _, out = tlk.spr_scores(s, tg)
        return tlk.launch_count() - before, out

    few, _ = launches(targets[:2])
    every, out = launches(targets)
    assert few == every
    many = np.resize(targets, 70000).astype(np.int32)
    n, out_many = launches(many)
    assert n == every + 1
    assert np.array_equal(out_many, out[np.arange(70000) % len(targets)])
    tlk.close()


def test_refusals():
    pb = branch_problem(4, 9, 50, 2, 260)
    tlk = make(pb)
    r = int(pb.root)
    for bad in (r, int(pb.left[r]), int(pb.right[r]), -1, pb.nnodes):
        with pytest.raises(phb.PhysherB200Error, match=r"^\[-1\]"):
            tlk.spr_targets(bad)
        with pytest.raises(phb.PhysherB200Error, match=r"^\[-1\]"):
            tlk.spr_scores(bad, [0])
    s = min((n for n in prunable(pb) if pb.left[n] >= 0), key=lambda n: ntips(pb, n))
    targets = tlk.spr_targets(s)
    assert len(targets) >= 4
    for e in (int(pb.parent[s]), r, s, int(pb.left[s]), -1, pb.nnodes):
        bad = targets.copy()
        bad[3] = e
        with pytest.raises(phb.PhysherB200Error, match=r"^\[-1\].*target 3"):
            tlk.spr_scores(s, bad)
    with pytest.raises(phb.PhysherB200Error, match=r"^\[-1\]"):
        tlk.spr_scores(s, targets[:0])
    with pytest.raises(phb.PhysherB200Error, match=r"^\[-1\].*target 0"):
        tlk.spr_scores(s, targets[:1], [-0.1])
    assert tlk.lib.phb_tlk_spr_scores(tlk.h, s, 1, None, None, None, None) == -1
    one = np.array(targets[:1], np.int32)
    assert tlk.lib.phb_tlk_spr_scores(tlk.h, s, 1, one.ctypes.data_as(_ip), None, None, None) == -1
    # the object still works
    lnl, out = tlk.spr_scores(s, targets)
    check(out, oracle_scores(pb, s, targets))
    assert rel_err(lnl, O.evaluate(pb, gradient=False)["lnl"]) < RTOL
    tlk.gradient()
    Pm, dPm = tlk.get_matrices()
    tlk.set_matrices(Pm, dPm)
    with pytest.raises(phb.PhysherB200Error, match=r"^\[-4\]"):
        tlk.spr_scores(s, targets)
    tlk.close()
