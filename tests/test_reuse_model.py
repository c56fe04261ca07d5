"""CPU: the plain-Python statement of tree reuse between moves (tests/sb_reuse_model.py) on records of the C oracle's games:
what is kept, in which order and with which links, what the next read-out sees, and every case that starts fresh."""
import numpy as np
import pytest

import sb_determinize_model as D
import sb_ismcts_model as I
import sb_oracle as O
import sb_reuse_model as R
import sb_search_model as M
from test_search_model import hash_eval, position


def searched(oracle, seed, plies, sims=48):
    """a finished perfect-information search of `sims` simulations from game `seed` after `plies` random plies"""
    tree = M.TreeModel(position(oracle, seed, plies), sims + 1)
    prior, value = hash_eval(tree.begin())
    for _ in range(sims):
        prior, value = hash_eval(tree.simulate(prior, value, 1.25, 0.0))
    result = tree.end(prior, value)
    return tree, result


def subtree(nodes, j):
    """node j and its descendants, in creation order"""
    inside = {j}
    for k in range(j + 1, len(nodes)):
        if nodes[k].parent in inside:
            inside.add(k)
    return sorted(inside)


def check_links(t):
    """parent < index, every child link points at a node whose parent is the linking node, and every non-root node is linked"""
    assert t.nodes[0].parent == -1
    linked = set()
    for k, nd in enumerate(t.nodes):
        if k:
            assert 0 <= nd.parent < k
        for c in nd.children.values():
            assert 0 < c < len(t.nodes) and t.nodes[c].parent == k
            linked.add(c)
    assert linked == set(range(1, len(t.nodes)))


def test_no_match_is_begin(oracle):
    src, _ = searched(oracle, 1, 6)
    other = position(oracle, 2, 6)
    t, leaf, kept = R.search_advance(src, other, 49, 49)
    fresh = M.TreeModel(other, 49)
    want = fresh.begin()
    assert kept == 0 and len(t.nodes) == 1 and (t.leaf, t.kind) == (fresh.leaf, fresh.kind)
    for a, b in zip(leaf, want):
        assert np.array_equal(np.asarray(a), np.asarray(b))
    # a source that is not finished (a leaf pending) or that was built for another max_steps starts fresh too
    t2 = M.TreeModel(src.root, 49)
    hash_eval(t2.begin())
    assert R.search_advance(t2, src.root, 49, 49)[2] == 0
    assert R.search_advance(src, src.root, 49, 49, max_steps=300)[2] == 0
    assert R.search_advance(None, src.root, 49, 49)[2] == 0


@pytest.mark.parametrize("seed", [0, 3, 5])
def test_child_of_the_played_action_keeps_its_subtree(oracle, seed):
    src, (visits, _q, _v) = searched(oracle, seed, 4 * seed)
    a = int(np.argmax(visits))
    c = src.nodes[0].children[a]
    nxt = O.step(src.root.copy(), a)
    assert nxt.tobytes() == src.nodes[c].rec.tobytes()  # the child's record is sb_step's
    order = subtree(src.nodes, c)
    t, leaf, kept = R.search_advance(src, nxt, 49 + 16, 10**6)
    assert kept == len(order) == len(t.nodes) and kept > 1
    new_index = {old: new for new, old in enumerate(order)}
    for new, old in enumerate(order):
        a_, b_ = t.nodes[new], src.nodes[old]
        assert a_.rec.tobytes() == b_.rec.tobytes() and (a_.N, a_.W, a_.terminal, a_.seat) == (b_.N, b_.W, b_.terminal, b_.seat)
        assert np.array_equal(a_.prior, b_.prior) and np.array_equal(a_.mask, b_.mask)
        assert a_.parent == (new_index[b_.parent] if new else -1)
        assert a_.children == {x: new_index[y] for x, y in b_.children.items()}
    check_links(t)
    assert leaf[0].tobytes() == nxt.tobytes() and leaf[5] == (M.TERMINAL if t.nodes[0].terminal else M.EVAL)
    want = M.TreeModel(nxt, 65).begin()
    for x, y in zip(leaf, want):
        assert np.array_equal(np.asarray(x), np.asarray(y))


def test_end_right_after_an_advance_reads_the_old_childs_children(oracle):
    src, (visits, _q, _v) = searched(oracle, 4, 9)
    a = int(np.argmax(visits))
    c = src.nodes[0].children[a]
    old = src.nodes[c]
    t, leaf, kept = R.search_advance(src, O.step(src.root.copy(), a), 65, 65)
    prior, value = hash_eval(leaf)
    v2, q2, rv2 = t.end(prior, value)
    sgn = M.sign(old.seat)
    for act in range(M.N_ACTIONS):
        cc = old.children.get(act)
        if cc is None:
            assert v2[act] == 0 and np.isnan(q2[act])
        else:
            assert v2[act] == src.nodes[cc].N and q2[act] == (sgn * src.nodes[cc].W) / float(src.nodes[cc].N)
    # the root gained this one evaluation, with the caller's prior replacing the stored one
    w = old.W + M.sign(old.seat) * float(np.float32(value))
    assert t.nodes[0].N == old.N + 1 and rv2 == (sgn * w) / float(old.N + 1)
    assert np.array_equal(t.nodes[0].prior, prior)


@pytest.mark.parametrize("keep", [1, 2, 5, 17, 64])
def test_keep_gives_a_connected_prefix(oracle, keep):
    src, (visits, _q, _v) = searched(oracle, 6, 3, sims=64)
    a = int(np.argmax(visits))
    c = src.nodes[0].children[a]
    order = subtree(src.nodes, c)
    t, _leaf, kept = R.search_advance(src, src.nodes[c].rec, 65, keep)
    assert kept == min(keep, len(order)) == len(t.nodes)
    assert [nd.rec.tobytes() for nd in t.nodes] == [src.nodes[k].rec.tobytes() for k in order[:kept]]
    check_links(t)
    # the same root again keeps the whole tree (continue searching), cut at keep
    t0, _leaf, kept0 = R.search_advance(src, src.root, 65, keep)
    assert kept0 == min(keep, len(src.nodes))
    check_links(t0)


def test_equal_records_pick_the_lowest_index(oracle):
    src, _ = searched(oracle, 7, 5)
    lo, hi = 3, len(src.nodes) - 2
    src.nodes[hi].rec = src.nodes[lo].rec.copy()
    assert R.search_match(src, src.nodes[lo].rec) == lo
    t, _leaf, _kept = R.search_advance(src, src.nodes[lo].rec, 49, 49)
    assert t.nodes[0].N == src.nodes[lo].N


def continued(oracle, t, leaf, sims):
    """S more simulations on an advanced tree; the root's visits then count the kept ones plus S + 1"""
    n0 = t.nodes[0].N
    prior, value = hash_eval(leaf)
    for _ in range(sims):
        prior, value = hash_eval(t.simulate(prior, value, 1.25, 0.0))
    visits, _q, _v = t.end(prior, value)
    assert t.nodes[0].N == n0 + sims + 1
    return visits


def test_an_advanced_tree_searches_on(oracle):
    src, (visits, _q, _v) = searched(oracle, 8, 6, sims=32)
    a = int(np.argmax(visits))
    c = src.nodes[0].children[a]
    whole = len(subtree(src.nodes, c))
    for keep in (whole, 3):
        t, leaf, kept = R.search_advance(src, O.step(src.root.copy(), a), 32 + 1 + 32, keep)
        assert kept == min(keep, whole) and kept > 1 and not t.nodes[0].terminal
        v = continued(oracle, t, leaf, 32)
        # the root was evaluated twice (as the child, and again as the new root); dropped nodes' visits still count in N
        assert v.sum() + 2 == t.nodes[0].N if keep == whole else v.sum() + 2 < t.nodes[0].N
        assert len(t.nodes) <= 65


# ---------------------------------------------------------------------------------------------- 8.8
def keys(count, salt):
    return (np.arange(count, dtype=np.uint64) * np.uint64(0x9E3779B97F4A7C15) + np.uint64(salt * 7919 + 1)).tolist()


def is_searched(root, sims, salt, max_nodes=None):
    t = I.ISTreeModel(max_nodes or sims + 1)
    ks = keys(sims + 1, salt)
    prior, value = hash_eval(t.begin(D.determinize(root, ks[0])))
    for k in range(1, sims + 1):
        prior, value = hash_eval(t.simulate(D.determinize(root, ks[k]), prior, value, 1.25, 0.0))
    visits, _q, _v = t.end(prior, value)
    return t, visits


def is_case(oracle):
    """(root, source tree, played, next root): a played action other than PASS after which the same seat is to move"""
    for seed in range(40):
        root = position(oracle, seed, 3 + seed % 7)
        if M.over(root, 400):
            continue
        t, visits = is_searched(root, 32, seed)
        a = int(np.argmax(visits))
        nxt = O.step(root.copy(), a)
        if M.seat(nxt) == M.seat(root) and not M.over(nxt, 400) and a != 155:
            return root, t, a, nxt
    raise AssertionError("no such position")


def test_ismcts_keeps_the_played_childs_subtree(oracle):
    root, src, a, nxt = is_case(oracle)
    c = src.nodes[0].children[src.root_code[a]]
    order = subtree(src.nodes, c)
    world = D.determinize(nxt, 12345)
    t, leaf, kept = R.ismcts_advance(src, world, a, 33 + 8, 10**6)
    assert kept == len(order) == len(t.nodes) and kept >= 1
    new_index = {old: new for new, old in enumerate(order)}
    for new, old in enumerate(order):
        x, y = t.nodes[new], src.nodes[old]
        assert (x.N, x.W, x.seat) == (y.N, y.W, y.seat) and np.array_equal(x.prior, y.prior)
        assert x.code == (I.NONE_CODE if new == 0 else y.code)
        assert x.children == {k: new_index[v] for k, v in y.children.items()}
    check_links(t)
    fresh = I.ISTreeModel(41)
    want = fresh.begin(world)
    for p, q in zip(leaf, want):
        assert np.array_equal(np.asarray(p), np.asarray(q))
    assert t.root_code == fresh.root_code and t.kind == M.EVAL
    # the tree searches on in fresh worlds of the new root
    prior, value = hash_eval(leaf)
    for k, key in enumerate(keys(8, 99)):
        prior, value = hash_eval(t.simulate(D.determinize(nxt, key), prior, value, 1.25, 0.0))
    t.end(prior, value)
    assert t.nodes[0].N == src.nodes[c].N + 9


def test_ismcts_falls_back(oracle):
    root, src, a, nxt = is_case(oracle)
    world = D.determinize(nxt, 777)
    assert R.ismcts_advance(src, world, a, 41, 41)[2] > 0
    fresh = I.ISTreeModel(41)
    want = fresh.begin(world)

    def fresh_like(played, w=world, s=src, max_steps=400):
        t, leaf, kept = R.ismcts_advance(s, w, played, 41, 41, max_steps)
        assert kept == 0 and len(t.nodes) == 1
        return leaf

    for leaf in (fresh_like(-1), fresh_like(156), fresh_like(255)):
        for p, q in zip(leaf, want):
            assert np.array_equal(np.asarray(p), np.asarray(q))
    illegal = [x for x in range(155) if src.root_code[x] == I.NONE_CODE]
    fresh_like(illegal[0])
    missing = [x for x in range(156) if src.root_code[x] != I.NONE_CODE and src.root_code[x] not in src.nodes[0].children]
    if missing:
        fresh_like(missing[0])
    small, vis = is_searched(root, 2, 5)  # two simulations: most codes have no child
    gone = [x for x in range(156) if small.root_code[x] != I.NONE_CODE and small.root_code[x] not in small.nodes[0].children]
    assert gone
    fresh_like(gone[0], s=small)
    # PASS hands the turn over: the new root's player is not the source root's, even where the PASS child's seat is its
    passes = 0
    for seed in range(12):
        r = position(oracle, seed, 5 + seed)
        if M.over(r, 400):
            continue
        s, _v = is_searched(r, 32, 40 + seed)
        if s.root_code[155] == I.PASS_CODE and I.PASS_CODE in s.nodes[0].children:
            pw = D.determinize(O.step(r.copy(), 155), 5)
            assert M.seat(pw) != M.seat(r) and s.nodes[s.nodes[0].children[I.PASS_CODE]].seat == M.seat(pw)
            fresh_like(155, w=pw, s=s)
            passes += 1
    assert passes >= 3
    # a world whose seat to move is not the child's, and a world that is over (FIRST's base below 0)
    flipped = world.copy()
    M.fields(flipped)["player_sign"] = -int(M.fields(flipped)["player_sign"])
    assert M.seat(flipped) != M.seat(world)
    fresh_like(a, w=flipped)
    ended = world.copy()
    M.fields(ended)["pl"][0]["base"] = -1
    assert M.over(ended, 400) and M.seat(ended) == M.seat(world)
    fresh_like(a, w=ended)
    # a source that was not finished
    pending = I.ISTreeModel(41)
    pending.begin(D.determinize(root, 1))
    fresh_like(a, s=pending)
    # a source built for another max_steps
    t, _leaf, kept = R.ismcts_advance(src, world, a, 41, 41, 399)
    assert kept == 0
