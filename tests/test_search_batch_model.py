"""CPU: the plain-Python statement of several leaves per tree per call (tests/sb_search_batch_model.py) on the C oracle, the
host-only size of its workspace through the C ABI, and the kernels of the library."""
import subprocess

import numpy as np
import pytest

import sb_search_batch_model as B
import sb_search_model as M
from monsoon_b200.engine import DEFAULT_DECKS, DEFAULT_FACTIONS, deck_indices
from test_search_model import hash_eval
from test_stack_frames import cuobjdump

DECKS = [np.array(deck_indices(d), dtype=np.uint8) for d in DEFAULT_DECKS]


def position(oracle, seed, plies, expert=False):
    """a record after `plies` steps of the oracle's uniform-random agent (or of its expert agent) from game `seed`"""
    st = oracle.new_game(seed, DECKS[0], DECKS[1], *DEFAULT_FACTIONS)
    if expert:
        for _ in range(plies):
            if M.over(st, 400):
                break
            st = oracle.step(st, oracle.expert_action(st))
    elif plies:
        oracle.rollout_random(st, plies)
    return st


def roots(oracle):
    return [position(oracle, s, 3 * s, expert=s % 2 == 1) for s in range(8)]


def same_leaf(w, g):
    """two emitted leaves (record, obs, obs_err, mask, to_move, kind) are equal"""
    return (w[0].tobytes() == g[0].tobytes() and np.array_equal(w[1], g[1]) and np.array_equal(w[3], g[3])
            and (w[2], w[4], w[5]) == (g[2], g[4], g[5]))


def run_batch(tree, calls, evaluate, c_puct=1.25, fpu=0.0, vl=1.0):
    """begin, `calls` batch calls and the batch end; returns (every call's leaves, read-out, kinds of every call)"""
    L = tree.L
    first = tree.begin()
    p, v = evaluate(first)
    prior, value = np.zeros((L, M.N_ACTIONS), np.float32), np.zeros(L, np.float32)
    prior[0], value[0] = p, v
    calls_out = [[first]]
    for _ in range(calls):
        leaves = tree.simulate_batch(prior, value, c_puct, fpu, vl)
        assert not any(tree.V), "virtual visits are zero between calls"
        calls_out.append(leaves)
        pv = [evaluate(lf) for lf in leaves]
        prior, value = np.stack([x[0] for x in pv]), np.array([x[1] for x in pv], np.float32)
    return calls_out, tree.end_batch(prior, value)


@pytest.mark.parametrize("c_puct,fpu", [(1.25, 0.0), (3.0, -0.5)])
def test_one_leaf_per_call_is_the_plain_search(oracle, c_puct, fpu):
    sims = 24
    for st in roots(oracle):
        plain = M.TreeModel(st, sims + 1)
        want = [plain.begin()]
        p, v = hash_eval(want[-1])
        for _ in range(sims):
            want.append(plain.simulate(p, v, c_puct, fpu))
            p, v = hash_eval(want[-1])
        want_end = plain.end(p, v)
        got, got_end = run_batch(B.BatchTreeModel(st, sims + 1, 1), sims, hash_eval, c_puct, fpu, vl=2.0)
        for w, g in zip(want, [c[0] for c in got]):
            assert same_leaf(w, g)
        assert np.array_equal(want_end[0], got_end[0])
        assert np.array_equal(want_end[1], got_end[1], equal_nan=True) and want_end[2] == got_end[2]


@pytest.mark.parametrize("L,vl", [(2, 1.0), (7, 0.0), (16, 3.5)])
def test_root_visits_add_up(oracle, L, vl):
    calls = 4
    for st in roots(oracle):
        tree = B.BatchTreeModel(st, 1 + calls * L, L)
        out, (visits, _q, _rv) = run_batch(tree, calls, hash_eval, vl=vl)
        lost = sum(kind in (B.COLLISION, M.FULL) for leaves in out[1:] for *_x, kind in leaves)
        if tree.nodes[0].terminal:
            assert visits.sum() == 0 and tree.nodes[0].N == 1 + calls * L
        else:
            assert visits.sum() + lost == calls * L
            assert tree.nodes[0].N == 1 + visits.sum()
        for j, nd in enumerate(tree.nodes):  # every node is a real record after the call that took it
            assert isinstance(nd, M.Node), j
            if j:
                assert nd.rec.tobytes() == oracle.step(tree.nodes[nd.parent].rec.copy(), nd.action).tobytes()


def test_collisions_are_on_nodes_of_the_same_call(oracle):
    seen = 0
    for st in roots(oracle):
        tree = B.BatchTreeModel(st, 1 + 4 * 16, 16)
        first = tree.begin()
        p, v = hash_eval(first)
        prior, value = np.zeros((16, M.N_ACTIONS), np.float32), np.zeros(16, np.float32)
        prior[0], value[0] = p, v
        for _ in range(4):
            start = len(tree.nodes)
            leaves = tree.simulate_batch(prior, value, 1.25, 0.0, 1.0)
            taken = {k for k, kind in tree.slots if kind in (M.EVAL, M.TERMINAL) and k >= start}
            for k, kind in tree.slots:
                if kind == B.COLLISION:
                    seen += 1
                    assert k >= start and k in taken
            pv = [hash_eval(lf) for lf in leaves]
            prior, value = np.stack([x[0] for x in pv]), np.array([x[1] for x in pv], np.float32)
    assert seen > 0


def test_hand_checked_few_legal_actions(oracle):
    """a root with three legal actions (PASS among them), L = 6, equal priors, vl = 1, c_puct = 1, fpu = 0, value 0"""
    st = next(cand for seed in range(300) for plies in range(0, 30, 3)
              for cand in [position(oracle, seed, plies)]
              if not M.over(cand, 400)
              and len(M.legal_ids(oracle.legal_mask(cand))) == 3 and 155 in M.legal_ids(oracle.legal_mask(cand)))
    a0, a1, a2 = M.legal_ids(oracle.legal_mask(st))
    assert a2 == 155  # PASS is the highest id
    tree = B.BatchTreeModel(st, 10, 6)
    tree.begin()
    flat = np.full((6, M.N_ACTIONS), 0.5, np.float32)
    zero = np.zeros(6, np.float32)
    tree.simulate_batch(flat, zero, 1.0, 0.0, 1.0)
    # slot 0: N(root) = 1, V = 0: every child unvisited, q = fpu = 0, u = 0.5 each: a0 (lowest id), new node 1
    # slot 1: V(root) = 1, a0's child has n = V = 1, q = (0 - 1) / 1 = -1: a1 wins (q 0, u = 0.5 * sqrt 2), node 2
    # slot 2: a2 = PASS, node 3
    # slot 3: sqrt(1 + 3) = 2; each child n = 1, q = -1, u = 0.5 * 2 / 2 = 0.5: all tie, a0 wins -> a pending node: COLLISION
    # slot 4: sqrt(1 + 4); a0's child n = V = 2, q = (0 - 2) / 2 = -1, u = 0.5 * sqrt 5 / 3; a1 and a2: q = -1,
    #         u = 0.5 * sqrt 5 / 2, larger: a1 -> COLLISION
    # slot 5: sqrt(1 + 5); a0 and a1 at n = 2, a2 at n = 1 has the larger u: a2 -> COLLISION
    kinds = [kind for _k, kind in tree.slots]
    nodes = [k for k, _kind in tree.slots]
    assert nodes == [1, 2, 3, 1, 2, 3], tree.slots
    assert kinds[3:] == [B.COLLISION] * 3 and all(kd in (M.EVAL, M.TERMINAL) for kd in kinds[:3])
    assert [tree.nodes[k].action for k in (1, 2, 3)] == [a0, a1, a2]
    visits, _q, _rv = tree.end_batch(flat, zero)
    assert visits[a0] == visits[a1] == visits[a2] == 1 and visits.sum() == 3 and tree.nodes[0].N == 4


def test_full_trees_give_full_slots(oracle):
    st = position(oracle, 2, 4)
    tree = B.BatchTreeModel(st, 5, 8)
    out, (visits, _q, _rv) = run_batch(tree, 3, hash_eval)
    assert len(tree.nodes) == 5
    assert [kind for *_x, kind in out[1]][4:] == [M.FULL] * 4
    assert all(kind == M.FULL for *_x, kind in out[2]) and all(kind == M.FULL for *_x, kind in out[3])
    assert visits.sum() == 4


def test_batch_workspace_bytes(built):
    from monsoon_b200 import _lib
    lib = _lib.load()
    for n, m, L in [(1, 1, 1), (3, 65, 16), (4096, 65, 16), (7, 17, 256), (0, 5, 3)]:
        tail = (8 * L + 4 * m + 15) // 16 * 16
        assert lib.sb_search_batch_workspace_bytes(n, m, L) == lib.sb_search_workspace_bytes(n, m) + n * tail
    for n, m, L in [(-1, 5, 1), (1, 0, 1), (1, 1 << 24 | 1, 1), (1, 5, 0), (1, 5, 257), (1, 5, -3), (1 << 30, 1 << 24, 256)]:
        assert lib.sb_search_batch_workspace_bytes(n, m, L) == 0, (n, m, L)


def test_batch_kernels_are_built(built):
    from monsoon_b200 import _lib
    out = subprocess.run([cuobjdump(), "-res-usage", _lib.SO_PATH], check=True, capture_output=True, text=True).stdout
    for name in ("k_search_batch_select", "k_search_batch_expand", "k_search_end_batch"):
        assert name in out, name


@pytest.fixture(scope="module")
def built():
    import __graft_entry__ as g
    g.build()
    return True
