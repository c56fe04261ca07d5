"""CPU: the plain-Python statement of several leaves per tree per call for the information-set search
(tests/sb_ismcts_batch_model.py) on the C oracle and sb_determinize_model's worlds -- one leaf per call is ISTreeModel, a
fixed world is the perfect-information batch model, a hand-worked collision case, the FULL cut-off in slot order -- the
host-only size of its workspace through the C ABI, and the new symbols of the library."""
import subprocess

import numpy as np
import pytest

import sb_determinize_model as D
import sb_ismcts_batch_model as IB
import sb_ismcts_model as I
import sb_search_batch_model as B
import sb_search_model as SM
from test_determinize_model import ended, hash_eval, keys, records
from test_search_batch_model import position
from test_stack_frames import cuobjdump


def live(step=9):
    return [st for st in records() if not ended(st)][::step]


def run_batch(tree, root, calls, salt, evaluate=hash_eval, c_puct=1.25, fpu=0.0, vl=1.0, fixed=False):
    """begin (world 0), `calls` batch calls over determinizations of root (or the root itself when fixed) and the batch
    end; returns (every call's leaves, read-out)"""
    L = tree.L
    ks = keys(1 + calls * L, salt)
    world = (lambda t: root.copy()) if fixed else (lambda t: D.determinize(root, ks[t]))
    first = tree.begin(world(0))
    p, v = evaluate(first)
    prior, value = np.zeros((L, SM.N_ACTIONS), np.float32), np.zeros(L, np.float32)
    prior[0], value[0] = p, v
    out = [[first]]
    for c in range(calls):
        leaves = tree.simulate_batch([world(1 + c * L + l) for l in range(L)], prior, value, c_puct, fpu, vl)
        assert len(leaves) == L and not any(tree.V), "virtual visits are zero between calls"
        out.append(leaves)
        pv = [evaluate(lf) for lf in leaves]
        prior, value = np.stack([x[0] for x in pv]), np.array([x[1] for x in pv], np.float32)
    return out, tree.end_batch(prior, value)


def same_leaf(w, g):
    return (w[0].tobytes() == g[0].tobytes() and np.array_equal(w[1], g[1]) and np.array_equal(w[3], g[3])
            and (w[2], w[4], w[5]) == (g[2], g[4], g[5]))


def same_end(a, b):
    return np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1], equal_nan=True) and (a[2] == b[2] or (a[2] != a[2] and b[2] != b[2]))


@pytest.mark.parametrize("c_puct,fpu", [(1.25, 0.0), (3.0, -0.5)])
def test_one_leaf_per_call_is_the_plain_search(oracle, c_puct, fpu):
    sims = 16
    for s, st in enumerate(live()):
        ks = keys(sims + 1, 40 + s)
        plain = I.ISTreeModel(sims + 1)
        want = [plain.begin(D.determinize(st, ks[0]))]
        for k in range(1, sims + 1):
            want.append(plain.simulate(D.determinize(st, ks[k]), *hash_eval(want[-1]), c_puct, fpu))
        want_end = plain.end(*hash_eval(want[-1]))
        got, got_end = run_batch(IB.ISBatchTreeModel(sims + 1, 1), st, sims, 40 + s, c_puct=c_puct, fpu=fpu, vl=2.5)
        assert all(same_leaf(w, g[0]) for w, g in zip(want, got)), s
        assert same_end(want_end, got_end), s


@pytest.mark.parametrize("L,vl", [(2, 1.0), (7, 0.0), (16, 3.5)])
def test_fixed_world_is_the_perfect_information_batch_search(oracle, L, vl):
    """every world is the root itself (default decks: no card twice in a hand): the leaves and read-out of
    sb_search_batch_model's BatchTreeModel"""
    calls = 3
    for s in range(8):
        st = position(oracle, s, 3 * s, expert=s % 2 == 1)
        pi = B.BatchTreeModel(st, 1 + calls * L, L)
        want = [[pi.begin()]]
        p, v = hash_eval(want[0][0])
        prior, value = np.zeros((L, SM.N_ACTIONS), np.float32), np.zeros(L, np.float32)
        prior[0], value[0] = p, v
        for _ in range(calls):
            want.append(pi.simulate_batch(prior, value, 1.25, 0.0, vl))
            pv = [hash_eval(lf) for lf in want[-1]]
            prior, value = np.stack([x[0] for x in pv]), np.array([x[1] for x in pv], np.float32)
        want_end = pi.end_batch(prior, value)
        got, got_end = run_batch(IB.ISBatchTreeModel(1 + calls * L, L), st, calls, 0, vl=vl, fixed=True)
        for c, (wc, gc) in enumerate(zip(want, got)):
            assert all(same_leaf(w, g) for w, g in zip(wc, gc)), (s, c)
        assert same_end(want_end, got_end), s


@pytest.mark.parametrize("L,vl", [(2, 1.0), (7, 0.0), (16, 3.5)])
def test_root_visits_add_up(oracle, L, vl):
    calls = 4
    for s, st in enumerate(live(23)):
        tree = IB.ISBatchTreeModel(1 + calls * L, L)
        out, (visits, _q, _rv) = run_batch(tree, st, calls, 60 + s, vl=vl)
        lost = sum(lf[5] in (IB.COLLISION, SM.FULL) for leaves in out[1:] for lf in leaves)
        assert visits.sum() + lost == calls * L, s
        assert tree.nodes[0].N == 1 + visits.sum()


def test_hand_checked_collisions_across_worlds(oracle):
    """a root with three legal representatives (PASS among them), L = 6, a different world per slot, equal priors, vl = 1,
    c_puct = 1, fpu = 0, value 0 (the same selections as sb_search_batch_model's hand-checked case: the root's legal set is
    the observer's own, the same in every world)"""
    st = next(cand for seed in range(300) for plies in range(0, 30, 3)
              for cand in [position(oracle, seed, plies)]
              if not SM.over(cand, 400) and len(I.representatives(cand)) == 3 and 155 in I.representatives(cand))
    a0, a1, a2 = I.representatives(st)
    ks = keys(7, 5)
    tree = IB.ISBatchTreeModel(10, 6)
    tree.begin(D.determinize(st, ks[0]))
    flat = np.full((6, SM.N_ACTIONS), 0.5, np.float32)
    zero = np.zeros(6, np.float32)
    worlds = [D.determinize(st, k) for k in ks[1:]]
    assert len({w.tobytes() for w in worlds}) == 6
    leaves = tree.simulate_batch(worlds, flat, zero, 1.0, 0.0, 1.0)
    # slot 0: N(root) = 1, V = 0: every id unvisited, q = fpu = 0, u = 0.5 each: a0 (lowest id), new node 1
    # slot 1: V(root) = 1, a0's child has n = V = 1, q = (0 - 1) / 1 = -1: a1 wins (q 0, u = 0.5 * sqrt 2), node 2
    # slot 2: a2 = PASS, node 3
    # slot 3: sqrt(1 + 3) = 2; each child n = 1, q = -1, u = 0.5 * 2 / 2 = 0.5: all tie, a0 wins -> a node of this call: COLLISION
    # slot 4: a0's child at n = 2 scores lower than a1's and a2's at n = 1: a1 -> COLLISION
    # slot 5: a0 and a1 at n = 2, a2 at n = 1 has the larger u: a2 -> COLLISION
    kinds = [kind for _k, kind, _t in tree.slots]
    assert [k for k, _kind, _t in tree.slots][:3] == [1, 2, 3], tree.slots
    assert kinds[3:] == [IB.COLLISION] * 3 and all(kd in (SM.EVAL, SM.TERMINAL) for kd in kinds[:3])
    h = I.hand(st)
    assert [tree.nodes[k].code for k in (1, 2, 3)] == [I.code(h, a) for a in (a0, a1, a2)]
    for l in range(3, 6):  # a collision emits its own world's root
        assert leaves[l][0].tobytes() == worlds[l].tobytes() and leaves[l][5] == IB.COLLISION
    for l in range(3):  # a new leaf is the world's record after the slot's action
        assert leaves[l][0].tobytes() == oracle.step(worlds[l].copy(), (a0, a1, a2)[l]).tobytes()
    visits, _q, _rv = tree.end_batch(flat, zero)
    assert visits[a0] == visits[a1] == visits[a2] == 1 and visits.sum() == 3 and tree.nodes[0].N == 4


def test_full_cut_off_in_slot_order(oracle):
    """max_nodes = 5, L = 8: the first slot that needs a node when none is free and every later slot are FULL, whatever
    the later slots would have reached; later calls stop the tree"""
    seen = 0
    for s, st in enumerate(live(31)):
        tree = IB.ISBatchTreeModel(5, 8)
        out, (visits, _q, _rv) = run_batch(tree, st, 3, 90 + s)
        calls = [[lf[5] for lf in leaves] for leaves in out[1:]]
        cut = next((c for c, kinds in enumerate(calls) if SM.FULL in kinds), None)
        if cut is None:
            continue
        kinds = calls[cut]
        full = kinds.index(SM.FULL)
        assert all(k == SM.FULL for k in kinds[full:]), (s, kinds)
        assert len(tree.nodes) == 5 and all(k == SM.FULL for kinds in calls[cut + 1:] for k in kinds), (s, calls)
        seen += full > 0
    assert seen > 0


def test_workspace_bytes(built):
    from monsoon_b200 import _lib
    lib = _lib.load()
    for n, m, L in [(1, 1, 1), (3, 65, 16), (4096, 65, 16), (7, 17, 256), (0, 5, 3)]:
        want = IB.workspace_bytes(n, m, L)
        assert want == lib.sb_ismcts_workspace_bytes(n, m) + n * ((16 * L + 4 * m + 15) // 16 * 16)
        assert lib.sb_ismcts_batch_workspace_bytes(n, m, L) == want, (n, m, L)
    for n, m, L in [(-1, 5, 1), (1, 0, 1), (1, 1 << 24 | 1, 1), (1, 5, 0), (1, 5, 257), (1, 5, -3), ((1 << 31) - 1, 1 << 24, 256)]:
        assert lib.sb_ismcts_batch_workspace_bytes(n, m, L) == 0, (n, m, L)
    from monsoon_b200.engine import ismcts_batch_workspace_bytes
    assert ismcts_batch_workspace_bytes(3, 65, 16) == IB.workspace_bytes(3, 65, 16)
    with pytest.raises(ValueError):
        ismcts_batch_workspace_bytes(3, 65, 257)


def test_new_symbols(built):
    from monsoon_b200 import _lib
    lib = _lib.load()
    for name in ("sb_ismcts_batch_workspace_bytes", "sb_ismcts_simulate_batch", "sb_ismcts_end_batch"):
        assert hasattr(lib, name), name
    out = subprocess.run([cuobjdump(), "-res-usage", _lib.SO_PATH], check=True, capture_output=True, text=True).stdout
    for name in ("k_ismcts_simulate_batch", "k_ismcts_end_batch"):
        assert name in out, name


@pytest.fixture(scope="module")
def built():
    import __graft_entry__ as g
    g.build()
    return True
