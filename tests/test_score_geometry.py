"""The score passes (calculate_branch, branch_hessian_diagonal's resident route, nni_scores, spr_scores) and the node-at-a-time
evaluation at the sizes where their launch geometry changes: state counts around each kernel's shared-memory thresholds (dynamic
shared memory past 48 KiB, the 512-thread SPR tile, the largest state count each call accepts), pattern counts around the 128- and
512-pattern tiles, item lists past one grid.y (65,535) on real trees, tip codes above S, and the refusal past each call's limit.

Reference values: the oracle (oracle.evaluate, oracle.branch_derivatives) on the exchanged or regrafted Problem (tests/test_nni.py,
tests/test_spr.py).  Tolerance: RTOL with the grad_err convention of tests/util.py.  Every case meant to cross a boundary asserts
that it did, from the launch counter or the item counts.
"""
import copy

import numpy as np
import pytest

import physher_b200 as phb
from oracle import oracle as O
from physher_b200 import synthetic as syn
from physher_b200.treelikelihood import KERNELS_GENERIC, OPT_INCREMENTAL, OPT_TUNE, RAN_GENERIC, RAN_TENSOR, RAN_WALK
from tests.test_branch import deriv_err
from tests.test_branch_hessian import branch_problem, make, oracle_hessian
from tests.test_nni import check, oracle_scores as nni_oracle
from tests.test_spr import oracle_scores as spr_oracle, prunable, prune_choices
from tests.util import RTOL, grad_err, rel_err

pytestmark = pytest.mark.gpu

GRID_Y = 65535  # items of one launch on grid.y


def smem_optin():
    import torch

    return int(torch.cuda.get_device_properties(0).shared_memory_per_block_optin)


def largest_s(nmat):
    """the largest state count whose nmat S x S double matrices fit one CTA's opt-in shared memory"""
    s = int(np.sqrt(smem_optin() / (8 * nmat)))
    while nmat * (s + 1) ** 2 * 8 <= smem_optin():
        s += 1
    while nmat * s * s * 8 > smem_optin():
        s -= 1
    return s


def fits(S, nmat):
    return nmat * S * S * 8 <= smem_optin()


def refusal(S, nmat):
    return rf"^\[-1\].*\b{S} states need {nmat * S * S * 8} bytes of shared memory"


def check_full(tlk, full):
    assert rel_err(tlk.calculate(), full["lnl"]) < RTOL
    assert grad_err(tlk.gradient(), full["grad"]) < RTOL


def branch_nodes(pb):
    """a tip and an internal node, neither the root"""
    return [next(n for n in range(pb.nnodes) if n != pb.root and pb.left[n] < 0),
            next(n for n in range(pb.nnodes) if n != pb.root and pb.left[n] >= 0)]


def launches(tlk, fn, *args):
    before = tlk.launch_count()
    out = fn(*args)
    return tlk.launch_count() - before, out


def sample(n, k, seed):
    """about k list positions: spread at random, plus 0, the last and the positions around the second grid.y slab"""
    pick = set(np.random.default_rng(seed).choice(n, size=min(n, k), replace=False).tolist()) | {0, n - 1}
    pick |= {p for p in (GRID_Y - 1, GRID_Y, GRID_Y + 1) if p < n}
    return np.array(sorted(pick))


def score_everything(pb, tlk, full, S):
    """calculate_branch, the Hessian diagonal, every NNI move and the SPR targets of a tip and an internal s, each against the oracle
    or refused past its shared-memory limit"""
    if fits(S, 3):
        for n in branch_nodes(pb):
            cands = pb.bl[n] * np.array([1.0, 0.3, 1.7])
            got = np.stack(tlk.calculate_branch(n, cands), 1)
            assert deriv_err(got, O.branch_derivatives(pb, n, cands)) < RTOL, n
        lnl, grad, hess = tlk.branch_hessian_diagonal()
        assert tlk.last_kernels() != RAN_WALK
        assert rel_err(lnl, full["lnl"]) < RTOL and grad_err(grad, full["grad"]) < RTOL
        assert grad_err(hess, oracle_hessian(pb)) < RTOL
    else:
        with pytest.raises(phb.PhysherB200Error, match=refusal(S, 3)):
            tlk.calculate_branch(0, [pb.bl[0]])
        with pytest.raises(phb.PhysherB200Error, match=refusal(S, 3)):
            tlk.branch_hessian_diagonal()
    moves = tlk.nni_moves()
    if fits(S, 4):
        lnl, out = tlk.nni_scores(moves)
        assert rel_err(lnl, full["lnl"]) < RTOL
        check(out, nni_oracle(pb, moves))
    else:
        with pytest.raises(phb.PhysherB200Error, match=refusal(S, 4)):
            tlk.nni_scores(moves)
    cand = prunable(pb)
    for s in (next(n for n in cand if pb.left[n] < 0), next(n for n in cand if pb.left[n] >= 0)):
        targets = tlk.spr_targets(s)
        if fits(S, 5):
            lnl, out = tlk.spr_scores(s, targets)
            assert rel_err(lnl, full["lnl"]) < RTOL
            check(out, spr_oracle(pb, s, targets))
        else:
            with pytest.raises(phb.PhysherB200Error, match=refusal(S, 5)):
                tlk.spr_scores(s, targets)
    check_full(tlk, full)  # the object still evaluates the current tree after every call and refusal


# ---------------------------------------------------------------------------------------------------------------------------------
# 1. state counts: around 48 KiB of dynamic shared memory for 2, 3, 4 and 5 matrices (S = 56 / 46 / 40 / 36), the 512-thread SPR tile
# (S >= 36), the pattern blocks of k_nni_operands (S <= 8 / <= 32 / > 32), the tensor-core state counts 60 ... 63 and their neighbours,
# and the largest state count each call accepts (read from the device: "max<nmat>" = the largest S whose nmat matrices fit).  35 states
# is a regression case: 49,000 bytes of dynamic shared memory for the SPR kernel's five matrices are under 48 KiB, but its 384 static
# bytes took the launch past the default limit without the opt-in
# ---------------------------------------------------------------------------------------------------------------------------------
SWEEP = [2, 3, 35, 36, 39, 40, 45, 46, 55, 56, 60, 62, 63, 64, 76, "max5", "max4", "max3", "max2"]


@pytest.mark.parametrize("C", [1, 3])
@pytest.mark.parametrize("S", SWEEP, ids=[str(s) for s in SWEEP])
def test_state_count_sweep(S, C):
    if isinstance(S, str):
        S = largest_s(int(S[3:]))
    T = 6 + S % 4  # 6 ... 9 tips
    pb = branch_problem(S, T, 129, C, 300 + S + C)
    assert np.any(pb.tip_states == S)  # some unknowns
    tlk = make(pb)
    full = O.evaluate(pb)
    check_full(tlk, full)
    score_everything(pb, tlk, full, S)
    tlk.close()


# ---------------------------------------------------------------------------------------------------------------------------------
# 2. pattern tiles: one pattern either side of 128 and 512 (k_branch_lnl, k_nni_score<4>, k_nni_contract, k_spr_score<4>: 128 threads;
# k_spr_score_any at S >= 36: 512; k_nni_operands: 128-pattern blocks at 20 states, 32 at 36 / 61), and one more than two 512 tiles
# ---------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("P", [127, 128, 129, 511, 512, 513, 1025])
@pytest.mark.parametrize("S,C", [(4, 2), (20, 4), (36, 1), (61, 4)], ids=["nuc4", "aa20", "s36", "codon61"])
def test_pattern_tiles(S, C, P):
    pb = branch_problem(S, 5, P, C, 400 + S + P)
    tlk = make(pb)
    full = O.evaluate(pb)
    check_full(tlk, full)
    score_everything(pb, tlk, full, S)
    tlk.close()


# ---------------------------------------------------------------------------------------------------------------------------------
# 3. item lists past one grid.y on random topologies (a caterpillar would take one evaluation launch per level)
# ---------------------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def big_trees():
    """T tips, 3 patterns (2 past 40,000 tips), one category: a random topology, lengths U(0.5, 5) / T and states evolved down the tree,
    so that every site likelihood stays far above 1e-154 (the oracle's d2 form, (L" L - L'^2) / L^2, underflows below it unscaled)"""
    cache = {}

    def get(S, T):
        if (S, T) not in cache:
            seed = 500 + S
            pb = branch_problem(S, 6, 3 if T < 40000 else 2, 1, seed)  # model and weights
            topo = syn.random_topology(T, seed)
            pb.left, pb.right, pb.parent, pb.root = topo.left, topo.right, topo.parent, topo.root
            pb.bl = syn.random_branch_lengths(topo, seed + 1, lo=0.5 / T, hi=5.0 / T, unrooted=False)
            pb.tip_states = syn.simulate_patterns(topo, pb.bl, pb.npatterns, S, seed + 2, unknown_frac=0.02)
            cache[(S, T)] = pb
        return cache[(S, T)]

    return get


@pytest.mark.parametrize("S,kernels", [(5, phb.KERNELS_AUTO), (4, KERNELS_GENERIC)], ids=["generic5", "nuc4-generic"])
def test_hessian_resident_route_past_one_launch(big_trees, S, kernels):
    pb = big_trees(S, 33000)
    n_items = pb.nnodes - 1
    assert n_items > GRID_Y + 1
    tlk = make(pb, kernels=kernels)
    lnl, grad, hess = tlk.branch_hessian_diagonal()
    assert tlk.last_kernels() == RAN_GENERIC
    # a repeat on clean resident partials: matrices, the score kernel once per grid.y slab, the sum; one slab more than one item
    n_all, (l2, g2, h2) = launches(tlk, tlk.branch_hessian_diagonal)
    n_one, _ = launches(tlk, tlk.calculate_branch, 0, [pb.bl[0]])
    print(f"Hessian diagonal of {n_items} branches: {n_all} launches, one branch: {n_one}")
    assert n_all == n_one + 1
    assert l2 == lnl and np.array_equal(g2, grad) and np.array_equal(h2, hess)
    full = O.evaluate(pb)
    assert rel_err(lnl, full["lnl"]) < RTOL
    assert grad_err(grad, full["grad"]) < RTOL
    g = tlk.gradient()  # the node-at-a-time gradient over the same > 65,535 branches
    assert grad_err(g, full["grad"]) < RTOL and grad_err(grad, g) < RTOL
    nodes = [n for n in range(pb.nnodes) if n != pb.root]  # the route's item list
    for k in sample(n_items, 16, 1):
        n = nodes[k]
        want = O.branch_derivatives(pb, n, [pb.bl[n]])[0]
        assert abs(hess[n] - want[2]) <= RTOL * max(abs(want[2]), 1e-6 * np.abs(hess).max()), n
    if S == 4:  # the fused 4-state walk (route 1) on the same inputs
        walk = make(pb)
        lw, gw, hw = walk.branch_hessian_diagonal()
        assert walk.last_kernels() == RAN_WALK
        assert rel_err(lw, lnl) < RTOL and grad_err(gw, grad) < RTOL and grad_err(hw, hess) < RTOL
        walk.close()
    tlk.close()


@pytest.mark.parametrize("S", [4, 5])
def test_spr_targets_past_one_launch(big_trees, S):
    pb = big_trees(S, 33000)
    tlk = make(pb)
    s = next(n for n in prunable(pb) if pb.left[n] < 0)  # a tip: 2(T - 1) - 3 targets in rooted mode
    targets = tlk.spr_targets(s)
    assert len(targets) == 2 * (pb.ntips - 1) - 3 and len(targets) > GRID_Y + 1
    tlk.spr_scores(s, targets[:2])
    n_two, _ = launches(tlk, tlk.spr_scores, s, targets[:2])
    n_all, (lnl, out) = launches(tlk, tlk.spr_scores, s, targets)
    print(f"SPR of tip {s}: {len(targets)} targets, {n_all} launches, 2 targets: {n_two}")
    assert n_all == n_two + 1
    assert rel_err(lnl, O.evaluate(pb, gradient=False)["lnl"]) < RTOL
    k = sample(len(targets), 16, 2)
    check(out[k], spr_oracle(pb, s, targets[k]))
    perm = np.random.default_rng(3).permutation(len(targets))
    _, shuffled = tlk.spr_scores(s, targets[perm])
    assert np.array_equal(shuffled, out[perm])
    tlk.close()


def test_nni_any_state_in_two_chunks(big_trees):
    """5 states: the operand chunk is capped at 65,535 moves, so 2(T - 2) > 65,535 moves take two chunks of two launches each"""
    pb = big_trees(5, 33000)
    tlk = make(pb)
    moves = tlk.nni_moves()
    assert len(moves) == 2 * (pb.ntips - 2) and len(moves) > GRID_Y + 1
    tlk.nni_scores(moves[:2])
    n_two, _ = launches(tlk, tlk.nni_scores, moves[:2])
    n_all, (lnl, out) = launches(tlk, tlk.nni_scores, moves)
    print(f"NNI, 5 states: {len(moves)} moves, {n_all} launches, 2 moves: {n_two}")
    assert n_all == n_two + 2
    assert rel_err(lnl, O.evaluate(pb, gradient=False)["lnl"]) < RTOL
    k = sample(len(moves), 16, 4)
    check(out[k], nni_oracle(pb, moves[k]))
    perm = np.random.default_rng(5).permutation(len(moves))
    _, shuffled = tlk.nni_scores(moves[perm])
    assert np.array_equal(shuffled, out[perm])
    tlk.close()


def test_nni_four_states_past_one_launch(big_trees):
    """k_nni_score<4> takes (v, x) groups on grid.y: more than 65,535 groups take a second launch"""
    pb = big_trees(4, 65600)
    tlk = make(pb)
    moves = tlk.nni_moves()
    groups = {(int(pb.parent[y]), int(x)) for x, y in moves}
    assert len(groups) > GRID_Y
    tlk.nni_scores(moves[:2])
    n_two, _ = launches(tlk, tlk.nni_scores, moves[:2])
    n_all, (lnl, out) = launches(tlk, tlk.nni_scores, moves)
    print(f"NNI, 4 states: {len(moves)} moves in {len(groups)} groups, {n_all} launches, 2 moves: {n_two}")
    assert n_all == n_two + 1
    assert rel_err(lnl, O.evaluate(pb, gradient=False)["lnl"]) < RTOL
    k = sample(len(moves), 16, 6)
    check(out[k], nni_oracle(pb, moves[k]))
    perm = np.random.default_rng(7).permutation(len(moves))
    _, shuffled = tlk.nni_scores(moves[perm])
    assert np.array_equal(shuffled, out[perm])
    tlk.close()


def test_branch_candidates_at_one_launch_and_one_more():
    """61 states: exactly 65,535 candidate lengths take one score launch, 65,536 two"""
    pb = branch_problem(61, 6, 3, 1, 600)
    tlk = make(pb)
    n = branch_nodes(pb)[1]
    cands = pb.bl[n] * np.linspace(0.2, 3.0, GRID_Y + 1)
    tlk.calculate_branch(n, cands[:2])
    n_one, head = launches(tlk, tlk.calculate_branch, n, cands[:GRID_Y])
    n_two, out = launches(tlk, tlk.calculate_branch, n, cands)
    print(f"calculate_branch, 61 states: {GRID_Y} candidates {n_one} launches, {GRID_Y + 1}: {n_two}")
    assert n_two == n_one + 1
    head, out = np.stack(head, 1), np.stack(out, 1)
    assert np.array_equal(out[:GRID_Y], head)
    k = sample(len(cands), 16, 8)
    assert deriv_err(out[k], O.branch_derivatives(pb, n, cands[k])) < RTOL
    perm = np.random.default_rng(9).permutation(len(cands))
    assert np.array_equal(np.stack(tlk.calculate_branch(n, cands[perm]), 1), out[perm])
    tlk.close()


# ---------------------------------------------------------------------------------------------------------------------------------
# 4. tip codes above S are unknown states, like the code S itself: every entry point gives the same bits
# ---------------------------------------------------------------------------------------------------------------------------------
def every_answer(pb, kernels, tune):
    """the answers of every entry point on a fresh object: a list of arrays"""
    out = []

    def fresh(k=kernels):
        t = make(pb, kernels=k)
        if tune:
            t.set_option(OPT_TUNE, tune)
        return t

    t = fresh()
    out += [np.array([t.calculate()]), t.pattern_log_likelihoods(), t.gradient()]
    family = t.last_kernels()
    bl = np.stack([pb.bl, pb.bl * 1.2])
    out += list(t.gradient_batch(bl))
    M = np.random.default_rng(10).uniform(-0.1, 0.1, (2, pb.nnodes, pb.ncat, pb.nstate, pb.nstate))
    out.append(t.matrix_gradient(M))
    t.close()
    for k in (kernels, KERNELS_GENERIC):  # the Hessian on both routes (the walk route at 4 states)
        t = fresh(k)
        out += list(t.branch_hessian_diagonal()[1:])
        t.close()
    t = fresh()
    for n in branch_nodes(pb):
        out += list(t.calculate_branch(n, pb.bl[n] * np.array([1.0, 0.5, 2.0])))
    out.append(t.nni_scores()[1])
    for s in prune_choices(pb)[:2]:
        out.append(t.spr_scores(s)[1])
    t.close()
    return out, family


@pytest.mark.parametrize("S,kernels,tune,family", [
    (4, phb.KERNELS_AUTO, 0, RAN_WALK), (20, phb.KERNELS_AUTO, 0, RAN_TENSOR), (61, phb.KERNELS_AUTO, 20, RAN_TENSOR),
    (61, phb.KERNELS_AUTO, 21, RAN_TENSOR), (5, phb.KERNELS_AUTO, 0, RAN_GENERIC)],
    ids=["nuc4-walk", "aa20-tensor-walk", "codon61-cherries", "codon61-no-cherries", "generic5"])
def test_unknown_codes_above_s(S, kernels, tune, family):
    pb = branch_problem(S, 9, 300, 2, 700 + S)
    unknown = pb.tip_states == S
    assert unknown.sum() >= 20
    other = copy.copy(pb)
    codes = np.array([c for c in (S + 1, 16, 255) if c > S], np.uint8)
    other.tip_states = pb.tip_states.copy()
    other.tip_states[unknown] = codes[np.arange(unknown.sum()) % len(codes)]
    want, fam = every_answer(pb, kernels, tune)
    assert fam == family
    assert rel_err(want[0][0], O.evaluate(pb, gradient=False)["lnl"]) < RTOL
    got, _ = every_answer(other, kernels, tune)
    assert len(got) == len(want)
    for i, (g, w) in enumerate(zip(got, want)):
        assert np.array_equal(g, w), i


# ---------------------------------------------------------------------------------------------------------------------------------
# 5. past each call's shared-memory limit: PHB_EINVAL naming the state count and the bytes, refused before any launch, the object still
# usable for everything else
# ---------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("nmat", [3, 4, 5], ids=["branch", "nni", "spr"])
def test_score_pass_refused_past_its_limit(nmat):
    S = largest_s(nmat) + 1
    assert fits(S, 2)  # the evaluation itself runs
    pb = branch_problem(S, 7, 64, 2, 800 + S)
    tlk = make(pb)
    full = O.evaluate(pb)
    tlk.update_uppers()  # resident partials in place: a refused call launches nothing at all
    calls = {3: [lambda: tlk.calculate_branch(0, [pb.bl[0]]), tlk.branch_hessian_diagonal], 4: [tlk.nni_scores],
             5: [lambda: tlk.spr_scores(prune_choices(pb)[0])]}[nmat]
    for call in calls:
        before = tlk.launch_count()
        with pytest.raises(phb.PhysherB200Error, match=refusal(S, nmat)):
            call()
        assert tlk.launch_count() == before
        check_full(tlk, full)
    tlk.close()


@pytest.mark.parametrize("S", ["max2+1", 255])
def test_evaluation_refused_past_its_limit(S):
    S = largest_s(2) + 1 if S == "max2+1" else S
    assert not fits(S, 2)
    pb = branch_problem(S, 5, 16, 1, 900)
    for kernels in (phb.KERNELS_AUTO, KERNELS_GENERIC):
        tlk = make(pb, kernels=kernels)
        M = np.zeros((1, pb.nnodes, pb.ncat, S, S))
        for call, nmat in ((tlk.calculate, 2), (tlk.gradient, 2), (tlk.pattern_log_likelihoods, 2), (lambda: tlk.matrix_gradient(M), 2),
                           (tlk.branch_hessian_diagonal, 3), (tlk.nni_scores, 4)):  # the score calls check their own, larger need first
            before = tlk.launch_count()
            with pytest.raises(phb.PhysherB200Error, match=refusal(S, nmat)):
                call()
            assert tlk.launch_count() == before
        tlk.set_option(OPT_INCREMENTAL, 1)
        with pytest.raises(phb.PhysherB200Error, match=refusal(S, 2)):
            tlk.calculate()
        tlk.close()
