"""CPU: the plain-Python search model (tests/sb_search_model.py) on the C oracle, the host-only workspace size of the C ABI,
and the torch helpers of monsoon_b200.search."""
import numpy as np
import pytest
import torch

import sb_search_model as M
from sb_env_model import EnvModel
from monsoon_b200.engine import DEFAULT_DECKS, DEFAULT_FACTIONS, deck_indices

DECKS = [np.array(deck_indices(d), dtype=np.uint8) for d in DEFAULT_DECKS]


def position(oracle, seed, plies):
    """a record after `plies` steps of the oracle's uniform-random agent from game `seed`"""
    st = oracle.new_game(seed, DECKS[0], DECKS[1], *DEFAULT_FACTIONS)
    if plies:
        oracle.rollout_random(st, plies)
    return st


def hash_eval(leaf):
    """a deterministic evaluator of the leaf record: prior from a hash of (digest, action), value in (-1, 1)"""
    import sb_oracle
    d = sb_oracle.digest(leaf[0])
    a = np.arange(M.N_ACTIONS, dtype=np.uint64)
    with np.errstate(over="ignore"):
        h = (np.uint64(d) ^ (a * np.uint64(0x9E3779B97F4A7C15))) * np.uint64(0xBF58476D1CE4E5B9)
    prior = ((h >> np.uint64(40)).astype(np.float64) / 2.0**24).astype(np.float32)
    return prior, np.float32(((d >> 11) % 2001) / 1000.0 - 1.0)


def run(tree, sims, evaluate, c_puct=1.25, fpu=0.0):
    leaves = [tree.begin()]
    prior, value = evaluate(leaves[-1])
    for _ in range(sims):
        leaves.append(tree.simulate(prior, value, c_puct, fpu))
        prior, value = evaluate(leaves[-1])
    return leaves, tree.end(prior, value)


def depth(tree, j):
    d = 0
    while tree.nodes[j].parent >= 0:
        j, d = tree.nodes[j].parent, d + 1
    return d


@pytest.mark.parametrize("c_puct,fpu", [(1.25, 0.0), (3.0, -0.5)])
def test_visit_counts_and_transitions(oracle, c_puct, fpu):
    sims = 40
    for seed in range(6):
        tree = M.TreeModel(position(oracle, seed, 7 * seed), sims + 1)
        leaves, (visits, q, root_value) = run(tree, sims, hash_eval, c_puct, fpu)
        root = tree.nodes[0]
        assert root.N == sims + 1 and visits.sum() == sims
        for j, nd in enumerate(tree.nodes):
            if nd.children:
                assert not nd.terminal and sum(tree.nodes[c].N for c in nd.children.values()) == nd.N - 1, (seed, j)
            if j:
                parent = tree.nodes[nd.parent]
                assert nd.action in M.legal_ids(parent.mask)
                assert nd.rec.tobytes() == oracle.step(parent.rec.copy(), nd.action).tobytes(), (seed, j)
        for a in range(M.N_ACTIONS):
            c = root.children.get(a)
            assert (np.isnan(q[a]) and visits[a] == 0) if c is None else q[a] == M.sign(root.seat) * tree.nodes[c].W / tree.nodes[c].N
        assert root_value == M.sign(root.seat) * root.W / root.N
        assert all(kind in (M.EVAL, M.TERMINAL) for *_x, kind in leaves)


def test_ties_go_to_the_lowest_action_id(oracle):
    st = position(oracle, 3, 4)
    legal = M.legal_ids(oracle.legal_mask(st))
    assert len(legal) > 3
    tree = M.TreeModel(st, 4)
    tree.begin()
    flat = np.full(M.N_ACTIONS, 0.25, dtype=np.float32)
    for k in range(3):  # equal priors, every child unvisited or of equal value: the lowest unvisited id wins each time
        tree.simulate(flat, np.float32(0.0), 1.0, 0.0)
        assert sorted(tree.nodes[0].children) == legal[:k + 1]


def test_q_signs_across_turns(oracle):
    """every leaf evaluation says FIRST is ahead by 0.5 (value +0.5 when FIRST is to move, -0.5 when SECOND is): every edge
    then has q = +0.5 below a node where FIRST moves and -0.5 below a node where SECOND moves, within a turn and across PASS"""
    seen = set()
    prior = np.linspace(1, 0.5, M.N_ACTIONS, dtype=np.float32)
    for seed in range(4):
        tree = M.TreeModel(position(oracle, 40 + seed, 3 * seed), 81)
        # fpu far below every value: the search deepens the visited line through several turns
        run(tree, 80, lambda leaf: (prior, np.float32(0.5 if leaf[4] == 0 else -0.5)), 1.0, -10.0)
        ends = {j for j, nd in enumerate(tree.nodes) if nd.terminal}  # a game value of +-1 enters the sums below these
        for j in list(ends):
            while j >= 0:
                ends.add(j)
                j = tree.nodes[j].parent
        for j, nd in enumerate(tree.nodes):
            for a, c in nd.children.items():
                ch = tree.nodes[c]
                if c in ends:
                    continue
                assert M.sign(nd.seat) * ch.W / ch.N == (0.5 if nd.seat == 0 else -0.5), (seed, j, a)
                assert (ch.seat == nd.seat) == (a != 155), (seed, j, a)
                seen.add((nd.seat, a == 155))
    assert len(seen) == 4, seen  # both seats to move, with actions of the same turn and with PASS


def test_small_max_steps_makes_depth_two_terminal(oracle):
    st = position(oracle, 9, 6)
    steps = int(M.fields(st)["steps"])
    tree = M.TreeModel(st, 41, max_steps=steps + 2)
    leaves, (visits, _q, _v) = run(tree, 40, hash_eval)
    assert max(depth(tree, j) for j in range(len(tree.nodes))) == 2
    term = [j for j in range(len(tree.nodes)) if depth(tree, j) == 2]
    assert term and all(tree.nodes[j].terminal and tree.nodes[j].tval == 0 for j in term)
    assert all(not tree.nodes[j].terminal for j in range(len(tree.nodes)) if depth(tree, j) < 2)
    assert sum(kind == M.TERMINAL for *_x, kind in leaves) > 0 and visits.sum() == 40


def test_full_tree_stops(oracle):
    tree = M.TreeModel(position(oracle, 2, 0), 3)
    leaves, (visits, _q, _v) = run(tree, 6, hash_eval)
    assert [kind for *_x, kind in leaves][3:] == [M.FULL] * 4 and len(tree.nodes) == 3
    assert tree.nodes[0].N == 3 and visits.sum() == 2
    assert all(leaf[0].tobytes() == tree.root.tobytes() for leaf in leaves[3:])


def test_rollout_evaluator_matches_oracle_rollouts(oracle):
    seen = set()
    for seed in range(30):
        st = position(oracle, 100 + seed, seed)
        tree = M.TreeModel(st, 2)
        leaf = tree.begin()
        rec = leaf[0].copy()
        prior, value = M.rollout_eval(leaf)
        legal = M.legal_ids(oracle.legal_mask(st))
        assert prior.dtype == np.float32 and np.all(prior[legal] == np.float32(1) / np.float32(len(legal)))
        assert np.count_nonzero(prior) == len(legal)
        acts, _d, _m = oracle.rollout_random(rec, 400)  # the same rollout, then the game's result by the bases
        assert rec.tobytes() == leaf[0].tobytes()
        r = EnvModel.result(rec)
        want = 0 if r not in (0, 1) else (1 if r == M.seat(st) else -1)
        assert value == want, seed
        seen.add(int(value))
    assert seen == {-1, 1}, seen


def test_workspace_bytes_is_host_only_and_refuses_bad_sizes():
    import __graft_entry__ as g
    g.build()
    from monsoon_b200 import _lib
    from monsoon_b200.engine import search_workspace_bytes
    ws = _lib.load().sb_search_workspace_bytes
    assert ws(1, 1) == 16 + 1808 and ws(0, 65) == 0 and ws(4096, 65) == 4096 * (16 + 65 * 1808)
    for n in (1, 2, 7, 100):
        for m in (1, 2, 17, 65, 1000):
            b = ws(n, m)
            assert b > 0 and b >= ws(n, max(1, m - 1)) and b > ws(n - 1, m) and b % 16 == 0
    for n, m in ((-1, 5), (5, 0), (5, -3), (1, 2**24 + 1), (2**31 - 1, 2**24)):
        assert ws(n, m) == 0, (n, m)
        with pytest.raises(ValueError):
            search_workspace_bytes(n, m)
    assert search_workspace_bytes(3, 9) == ws(3, 9)


def test_select_actions_and_masked_softmax():
    from monsoon_b200.search import legal_actions, masked_softmax, select_actions
    v = torch.zeros((4, 156), dtype=torch.int32)
    v[0, [3, 9]] = 5
    v[1, 7] = 1
    v[3, [2, 150]] = torch.tensor([1, 40], dtype=torch.int32)
    assert select_actions(v).tolist() == [3, 7, 255, 150]
    g = torch.Generator().manual_seed(0)
    s = torch.stack([select_actions(v, 1.0, g) for _ in range(400)])
    assert set(s[:, 0].tolist()) == {3, 9} and set(s[:, 1].tolist()) == {7} and set(s[:, 2].tolist()) == {255}
    assert set(s[:, 3].tolist()) <= {2, 150} and (s[:, 3] == 150).sum() > 300
    masks = torch.zeros((2, 5), dtype=torch.int32)
    masks[0, 0] = 0b1010
    masks[1, 4] = 1 << (155 - 128)
    legal = legal_actions(masks)
    assert legal[0].nonzero().flatten().tolist() == [1, 3] and legal[1].nonzero().flatten().tolist() == [155]
    p = masked_softmax(torch.zeros((2, 156)), masks)
    assert p.dtype == torch.float32 and p[0, 1] == p[0, 3] == 0.5 and p[1, 155] == 1 and p.sum() == 2
