"""CPU: the plain-Python information-set search model (tests/sb_ismcts_model.py) on records of the C oracle's games -- move
codes, the root's codes in every world, visit sums, leaves that are oracle steps of the world's record, the tie to the
perfect-information model in a fixed world -- and the host-only workspace size of the C ABI."""
import numpy as np
import pytest

import sb_determinize_model as D
import sb_ismcts_model as I
import sb_search_model as SM
from test_determinize_model import ended, fields, hash_eval, keys, records


def live(step=5):
    return [st for st in records() if not ended(st)][::step]


def with_copy(st, src=0, dst=1):
    """st with the mover's hand slot dst holding a copy of slot src's (card, cost, flags)"""
    out = st.copy()
    f = fields(out)
    p = f["pl"][int(f["local_order"])]
    for nm in ("hand_card", "hand_cost", "hand_flags"):
        p[nm][dst] = p[nm][src]
    return out


def test_codes_follow_the_hand(oracle):
    """every legal id's code names its kind, the card in its slot and its target / swap partner"""
    n = 0
    for st in live():
        h = I.hand(st)
        for a in SM.legal_ids(oracle.legal_mask(st.copy())):
            c = I.code(h, a)
            kind, card, x = c >> 24, c >> 16 & 255, c & 0xFFFF
            if a < 64:
                assert (kind, card, x) == (0, h[a >> 4], a & 15)
            elif a < 148:
                assert (kind, card, x) == (1, h[(a - 64) // 21], (a - 64) % 21)
            elif a < 152:
                assert (kind, card, x) == (2, h[a - 148], 0)
            elif a < 155:
                assert (kind, card, x) == (3, h[a - 151], h[0])
            else:
                assert c == I.PASS_CODE
            n += 1
    assert n > 2000


def test_duplicate_cards_share_a_code(oracle):
    """with a copy of slot 0's card in slot 1, slot 1's ids take slot 0's codes and only the lower id represents each"""
    found = 0
    for st in live(3):
        d = with_copy(st)
        legal = SM.legal_ids(oracle.legal_mask(d.copy()))
        reps = I.representatives(d)
        h = I.hand(d)
        codes = [I.code(h, a) for a in reps]
        assert len(set(codes)) == len(codes) and set(codes) == {I.code(h, a) for a in legal}
        for a in legal:
            lo = [b for b in legal if b < a and I.code(h, b) == I.code(h, a)]
            assert (a in reps) == (not lo)
        dup = [a for a in legal if a not in reps]
        if dup:
            found += 1
            for a in dup:
                ci, first, stride = I.slot(a)
                assert ci >= 1 and a - stride in legal and I.code(h, a - stride) == I.code(h, a)
    assert found > 50, found


def test_root_codes_are_the_same_in_every_world(oracle):
    for g, st in enumerate(live(4)):
        want = I.ISTreeModel(2)
        want.begin(st)
        for key in keys(3, 300 + g):
            t = I.ISTreeModel(2)
            leaf = t.begin(D.determinize(st, key))
            assert t.root_code == want.root_code, g
            assert (int(fields(leaf[0])["seed_lo"]), int(fields(leaf[0])["seed_hi"])) == (key & D.M32, key >> 32)


def run(root, sims, salt, evaluate=hash_eval, c_puct=1.25, fpu=0.0, max_nodes=None, max_steps=400, fixed=False):
    """(tree, [(world, leaf)] per call, read-out): world k = determinize(root, key k), or the root itself when fixed"""
    t = I.ISTreeModel(max_nodes or sims + 1, max_steps)
    worlds = [root.copy() if fixed else D.determinize(root, k) for k in keys(sims + 1, salt)]
    calls = [(worlds[0], t.begin(worlds[0]))]
    prior, value = evaluate(calls[-1][1])
    for k in range(1, sims + 1):
        calls.append((worlds[k], t.simulate(worlds[k], prior, value, c_puct, fpu)))
        prior, value = evaluate(calls[-1][1])
    return t, calls, t.end(prior, value)


@pytest.mark.parametrize("c_puct,fpu", [(1.25, 0.0), (3.0, -0.5)])
def test_visit_sums_and_leaf_outputs(oracle, c_puct, fpu):
    """visits add up to the simulations, every leaf carries its world's key, its legal mask and seat"""
    sims = 24
    kinds = set()
    for g, st in enumerate(live(40)[:12]):
        t, calls, (visits, q, root_value) = run(st, sims, 700 + g, c_puct=c_puct, fpu=fpu)
        assert t.nodes[0].N == sims + 1 and visits.sum() == sims, g
        assert np.isnan(q[visits == 0]).all() and not np.isnan(q[visits > 0]).any()
        assert root_value == SM.sign(t.nodes[0].seat) * t.nodes[0].W / t.nodes[0].N
        for j, nd in enumerate(t.nodes):  # a walk can end at an existing node that is terminal in its world
            assert sum(t.nodes[c].N for c in nd.children.values()) <= nd.N - 1, (g, j)
        for k, (world, (rec, _obs, _err, mask, to_move, kind)) in enumerate(calls):
            kinds.add(kind)
            assert rec[:8].tobytes() == world[:8].tobytes(), (g, k)  # the world's key
            assert np.array_equal(mask, oracle.legal_mask(rec.copy()).view(np.int32)) and to_move == SM.seat(rec)
    assert SM.EVAL in kinds


def test_leaves_are_oracle_steps_of_the_world(oracle):
    """after each call the model's path holds, per node, the world's record there: the world's root, then one oracle step of
    the record above for the action id that has the node's code; the leaf is the last of them"""
    for g, st in enumerate(live(40)[:4]):
        t = I.ISTreeModel(33)
        for k, key in enumerate(keys(33, 91 + g)):
            w = D.determinize(st, key)
            leaf = t.begin(w) if k == 0 else t.simulate(w, *hash_eval(leaf), 1.25, 0.0)
            assert t.path[0][1].tobytes() == w.tobytes()
            for (pa, ra), (nb, rb) in zip(t.path, t.path[1:]):
                assert t.nodes[nb].parent == pa
                a = [b for b in I.representatives(ra) if I.code(I.hand(ra), b) == t.nodes[nb].code]
                assert len(a) == 1 and oracle.step(ra.copy(), a[0]).tobytes() == rb.tobytes(), (g, k)
            assert t.path[-1][1].tobytes() == leaf[0].tobytes()
        assert len(t.nodes) > 10


def no_duplicates(st):
    f = fields(st)
    return all(len(set(int(c) for c in p["hand_card"][:int(p["n_hand"])])) == int(p["n_hand"]) for p in f["pl"])


def test_fixed_world_equals_the_perfect_information_model(oracle):
    """with the root itself as every world (and no card twice in a hand), the search is sb_search_model's, call for call"""
    roots = [st for st in live(30) if no_duplicates(st)][:8]
    assert len(roots) >= 6
    for g, st in enumerate(roots):
        sims = 20
        t, calls, (visits, q, rv) = run(st, sims, 0, fixed=True)
        ref = SM.TreeModel(st, sims + 1)
        want = [ref.begin()]
        prior, value = hash_eval(want[-1])
        for _ in range(sims):
            want.append(ref.simulate(prior, value, 1.25, 0.0))
            prior, value = hash_eval(want[-1])
        wv, wq, wr = ref.end(prior, value)
        for k, ((_w, got), exp) in enumerate(zip(calls, want)):
            assert got[0].tobytes() == exp[0].tobytes() and got[5] == exp[5], (g, k)
        assert np.array_equal(visits, wv) and np.array_equal(q, wq, equal_nan=True) and rv == wr, g


def test_small_max_steps_and_full_trees(oracle):
    st = live(30)[2]
    steps = int(fields(st)["steps"])
    t, calls, (visits, _q, _v) = run(st, 24, 5, max_steps=steps + 2)
    assert any(kind == SM.TERMINAL for _w, (*_x, kind) in calls) and visits.sum() == 24
    t, calls, (visits, _q, _v) = run(st, 8, 6, max_nodes=4)
    kinds = [kind for _w, (*_x, kind) in calls]
    assert kinds[4:] == [SM.FULL] * 5 and len(t.nodes) == 4 and visits.sum() == 3
    assert all(leaf[0].tobytes() == w.tobytes() for w, leaf in calls[4:])  # the world's root is emitted


def test_workspace_bytes_is_host_only_and_refuses_bad_sizes():
    import __graft_entry__ as g
    g.build()
    from monsoon_b200 import _lib
    from monsoon_b200.engine import ismcts_workspace_bytes
    ws = _lib.load().sb_ismcts_workspace_bytes
    assert ws(1, 1) == 656 * 2 and ws(0, 65) == 0 and ws(4096, 65) == 4096 * 656 * 66
    for n in (0, 1, 2, 7, 100):
        for m in (1, 2, 17, 65, 1000):
            assert ws(n, m) == I.workspace_bytes(n, m) and ws(n, m) % 16 == 0
    for n, m in ((-1, 5), (5, 0), (5, -3), (1, 2**24 + 1), (2**31 - 1, 2**24)):
        assert ws(n, m) == 0, (n, m)
        with pytest.raises(ValueError):
            ismcts_workspace_bytes(n, m)
    assert ismcts_workspace_bytes(3, 9) == ws(3, 9)
    assert _lib.load().sb_abi_version() == 5
