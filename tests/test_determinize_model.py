"""CPU: the plain-Python statement of sb_determinize (tests/sb_determinize_model.py) on records of the C oracle's games --
what the observer sees is kept, what is hidden is resampled uniformly, the record still plays -- and the PIMC read-out."""
import functools
import os

import numpy as np
import pytest
from scipy.stats import chisquare

import sb_determinize_model as D
import sb_search_model as SM
from sb_layout import CF_OBJ, STATE_DTYPE
from monsoon_b200.engine import CARD_INDEX, DEFAULT_DECKS, DEFAULT_FACTIONS, deck_indices

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
DECKS = [np.array(deck_indices(d), dtype=np.uint8) for d in DEFAULT_DECKS]
TRIPLES = ("hand_card", "hand_cost", "hand_flags", "deck_card", "deck_cost", "deck_flags")


def fields(st):
    return st.view(STATE_DTYPE)[0]


def ended(st):
    f = fields(st)
    return bool(f["err"] or f["pl"][0]["base"] < 0 or f["pl"][1]["base"] < 0 or f["steps"] >= 400)


def play(oracle, st, plies, rs, expert):
    """records along one game: random legal actions (numpy stream) or the oracle's expert_action"""
    out = []
    for _ in range(plies):
        if ended(st):
            break
        a = oracle.expert_action(st) if expert else rs.choice(SM.legal_ids(oracle.legal_mask(st)))
        oracle.step(st, a)
        out.append(st.copy())
    return out


def games():
    """(seed, deck0, deck1, faction0, faction1) of default-deck, random-deck and focused-deck games"""
    rd = np.load(os.path.join(G, "randdeck_chain.npz"))
    cf = np.load(os.path.join(G, "card_focus.npz"))
    out = [(s, DECKS[0], DECKS[1], *DEFAULT_FACTIONS) for s in range(12)]
    out += [(int(rd["seeds"][i]), rd["decks"][i][0], rd["decks"][i][1], int(rd["factions"][i][0]), int(rd["factions"][i][1]))
            for i in range(0, 3000, 250)]
    out += [(int(cf["seeds"][i]), cf["decks"][i][0], cf["decks"][i][1], int(cf["factions"][i][0]), int(cf["factions"][i][1]))
            for i in range(0, 896, 75)]
    return out


@functools.lru_cache(maxsize=None)
def records():
    import sb_oracle as oracle
    oracle.build()
    rs = np.random.RandomState(5)
    out = []
    for g, (seed, d0, d1, f0, f1) in enumerate(games()):
        for expert in (False, True):
            st = oracle.new_game(seed, d0, d1, f0, f1)
            out.append(st.copy())
            out += play(oracle, st, 60, rs, expert)[::2]
    return out


def keys(count, salt):
    return [(salt * 0x9E3779B97F4A7C15 + 0xD1B54A32D192ED03 * (t + 1)) & D.M64 for t in range(count)]


def hash_eval(leaf):
    """a deterministic evaluator of a search-model leaf: prior from a hash of (digest, action), value in [-1, 1]"""
    import sb_oracle
    d = sb_oracle.digest(leaf[0])
    a = np.arange(SM.N_ACTIONS, dtype=np.uint64)
    with np.errstate(over="ignore"):
        h = (np.uint64(d) ^ (a * np.uint64(0x9E3779B97F4A7C15))) * np.uint64(0xBF58476D1CE4E5B9)
    return ((h >> np.uint64(40)).astype(np.float64) / 2.0**24).astype(np.float32), np.float32(((d >> 11) % 2001) / 1000.0 - 1.0)


def multiset(f, r):
    p = f["pl"][r]
    return sorted([tuple(int(x) for x in t) for t in zip(p["hand_card"][:p["n_hand"]], p["hand_cost"][:p["n_hand"]], p["hand_flags"][:p["n_hand"]])]
                  + [tuple(int(x) for x in t) for t in zip(p["deck_card"][:p["n_deck"]], p["deck_cost"][:p["n_deck"]], p["deck_flags"][:p["n_deck"]])])


def test_records_cover_both_seats_and_ends(oracle):
    recs = records()
    assert len(recs) > 1500
    assert {int(fields(st)["local_order"]) for st in recs} == {0, 1}
    assert any(ended(st) for st in recs)


def test_observer_view_is_invariant(oracle):
    """observation, legal mask and features of the default observer are those of the original record"""
    pairs = 0
    for g, st in enumerate(records()):
        obs, oerr = oracle.observe(st.copy())
        mask = oracle.legal_mask(st.copy())
        feat, ferr = oracle.features(st.copy())
        for key in keys(2, g):
            d = D.determinize(st, key)
            o2, e2 = oracle.observe(d.copy())
            f2, fe2 = oracle.features(d.copy())
            assert np.array_equal(obs, o2) and oerr == e2, g
            assert np.array_equal(mask, oracle.legal_mask(d.copy())), g
            assert np.array_equal(feat, f2, equal_nan=True) and ferr == fe2, g
            pairs += 1
    assert pairs >= 3000


def test_only_the_hidden_triples_and_the_key_change(oracle):
    changed_hand = total = 0
    for g, st in enumerate(records()):
        for observer in (None, 0, 1):
            f = fields(st)
            o = int(f["local_order"] != 0) if observer is None else observer
            r = 1 - o
            key = keys(1, 1000 + g)[0]
            d = D.determinize(st, key, observer)
            fd = fields(d)
            assert (int(fd["seed_lo"]), int(fd["seed_hi"])) == (key & D.M32, key >> 32)
            a, b = st.view(STATE_DTYPE).copy(), d.view(STATE_DTYPE).copy()
            for x in (a, b):
                x[0]["seed_lo"] = x[0]["seed_hi"] = 0
                for nm in TRIPLES:
                    x[0]["pl"][r][nm] = 0
            assert a.tobytes() == b.tobytes(), (g, observer)
            assert multiset(f, r) == multiset(fd, r) and multiset(f, o) == multiset(fd, o)
            assert fd["pl"][r]["n_hand"] == f["pl"][r]["n_hand"] and fd["pl"][r]["n_deck"] == f["pl"][r]["n_deck"]
            assert np.array_equal(fd["pl"][r]["deck_wn"], f["pl"][r]["deck_wn"])
            nh = int(f["pl"][r]["n_hand"])
            if nh and len(D.movable_slots(f, r)) > nh:
                total += 1
                changed_hand += sorted(f["pl"][r]["hand_card"][:nh].tolist()) != sorted(fd["pl"][r]["hand_card"][:nh].tolist())
    assert total > 1000 and changed_hand > total // 2, (changed_hand, total)  # the opponent's hand is resampled


def obj_records(oracle):
    """records of the focused B305 games in which a board instance of B305 sits in a hand or deck: (record, seat holding it)"""
    cf = np.load(os.path.join(G, "card_focus.npz"))
    rs = np.random.RandomState(9)
    out = []
    for i in np.flatnonzero(cf["card"] == CARD_INDEX["B305"]):
        for rep in range(6):
            st = oracle.new_game(int(cf["seeds"][i]) + 7919 * rep, cf["decks"][i][0], cf["decks"][i][1], int(cf["factions"][i][0]), int(cf["factions"][i][1]))
            for rec in play(oracle, st, 120, rs, rep % 2 == 1):
                f = fields(rec)
                for seat in (0, 1):
                    p = f["pl"][seat]
                    if (p["hand_flags"][:p["n_hand"]] & CF_OBJ).any() or (p["deck_flags"][:p["n_deck"]] & CF_OBJ).any():
                        out.append((rec, seat))
    return out


def test_board_instances_stay_put(oracle):
    found = obj_records(oracle)
    assert len(found) >= 5, len(found)
    for g, (st, seat) in enumerate(found):
        f = fields(st)
        p = f["pl"][seat]
        objs = [("hand", h) for h in range(p["n_hand"]) if p["hand_flags"][h] & CF_OBJ] + \
               [("deck", d) for d in range(p["n_deck"]) if p["deck_flags"][d] & CF_OBJ]
        for key in keys(8, 77 + g):
            d = D.determinize(st, key, observer=1 - seat)
            q = fields(d)["pl"][seat]
            for kind, i in objs:
                assert all(q[kind + nm][i] == p[kind + nm][i] for nm in ("_card", "_cost", "_flags")), (g, kind, i)
            assert multiset(f, seat) == multiset(fields(d), seat)
            o, e = oracle.observe(st.copy())
            o2, e2 = oracle.observe(D.determinize(st, key).copy())
            assert np.array_equal(o, o2) and e == e2


def test_determinized_records_play_on(oracle):
    """a determinized record plays to the end in the oracle.  Its statuses are rule statuses (codes 1-4: the reference raises
    there too, as it does in ordinary games) or this engine's capacity statuses (5-7), and they are no more frequent than in
    rollouts of the original records under the same new keys"""
    recs = [st for st in records() if not ended(st)][::3]
    assert len(recs) > 200
    orig, det = {}, {}
    for g, st in enumerate(recs):
        for key in keys(3, 5000 + g):
            a = st.copy()
            fa = fields(a)
            fa["seed_lo"], fa["seed_hi"] = key & D.M32, key >> 32
            oracle.rollout_random(a, 400)
            orig[int(a[18])] = orig.get(int(a[18]), 0) + 1
            b = D.determinize(st, key)
            _acts, dig, _m = oracle.rollout_random(b, 400)
            assert ended(b) and len(dig) > 0, g
            det[int(b[18])] = det.get(int(b[18]), 0) + 1
    assert set(det) <= set(range(8)), det  # SB_ERR_NONE .. SB_ERR_DEPTH
    bad_det, bad_orig = sum(det.values()) - det.get(0, 0), sum(orig.values()) - orig.get(0, 0)
    assert bad_det <= 2 * bad_orig + 10, (det, orig)


@pytest.mark.parametrize("nh,nd,obj", [(4, 8, ()), (3, 10, ()), (4, 9, (("deck", 2), ("hand", 1)))])
def test_slots_are_uniform(oracle, nh, nd, obj):
    """which slot each card lands in, over 20,000 fixed keys: chi-square against the uniform law (fixed keys: no flakes)"""
    st = records()[40].copy()
    f = fields(st)
    r = 1 - int(f["local_order"] != 0)
    p = f["pl"][r]
    p["n_hand"], p["n_deck"] = nh, nd
    p["hand_flags"][:] = 0
    p["deck_flags"][:] = 0
    for kind, i in obj:
        p[kind + "_flags"][i] = CF_OBJ
    p["hand_card"][:] = np.arange(1, 5)
    p["deck_card"][:] = np.arange(5, 21)
    slots = D.movable_slots(f, r)
    m = len(slots)
    assert m == nh + nd - len(obj)
    ids = [int(p["deck_card"][i] if d else p["hand_card"][i]) for d, i in slots]
    counts = np.zeros((m, m), dtype=np.int64)  # [card, position in the movable list]
    n = 20000
    for key in keys(n, 31 + m):
        q = fields(D.determinize(st, key))["pl"][r]
        for pos, (d, i) in enumerate(slots):
            counts[ids.index(int(q["deck_card"][i] if d else q["hand_card"][i])), pos] += 1
        for kind, i in obj:
            assert q[kind + "_card"][i] == p[kind + "_card"][i]
    assert (counts.sum(0) == n).all() and (counts.sum(1) == n).all()
    pv = [chisquare(counts[c]).pvalue for c in range(m)] + [chisquare(counts[:, s]).pvalue for s in range(m)]
    assert min(pv) > 1e-4 / len(pv), min(pv)


def test_pimc_readout_sums_and_weights(oracle):
    """K trees per root on determinized roots: the root legal set is the same in all K, visits add up, q is the visit-weighted
    mean of the per-tree q and the root value the mean of the per-tree root values"""
    n, k, sims = 3, 4, 24
    roots = [st for st in records() if not ended(st)][10:10 + n]
    trees = []
    for i, root in enumerate(roots):
        for s, key in enumerate(keys(k, 900 + i)):
            d = D.determinize(root, key)
            assert np.array_equal(oracle.legal_mask(d.copy()), oracle.legal_mask(root.copy()))
            trees.append(SM.TreeModel(d, sims + 1))
    leaves = [t.begin() for t in trees]
    for _ in range(sims):
        ev = [hash_eval(lf) for lf in leaves]
        leaves = [t.simulate(ev[g][0], ev[g][1], 1.25, 0.0) for g, t in enumerate(trees)]
    ev = [hash_eval(lf) for lf in leaves]
    prior, value = [e[0] for e in ev], [e[1] for e in ev]
    per = [SM.TreeModel.end(t, prior[g], value[g]) for g, t in enumerate(trees)]
    for t in trees:  # end() is idempotent once nothing is pending
        t.kind = SM.FULL
    visits, q, rv = D.pimc_readout(trees, prior, value, n, k)
    for i in range(n):
        vis = np.stack([per[i * k + s][0] for s in range(k)])
        assert np.array_equal(visits[i], vis.sum(0)) and visits[i].sum() == k * sims
        for a in range(SM.N_ACTIONS):
            if visits[i, a] == 0:
                assert np.isnan(q[i, a])
            else:
                want = sum(per[i * k + s][1][a] * vis[s, a] for s in range(k) if vis[s, a]) / visits[i, a]
                assert abs(q[i, a] - want) <= 1e-12
        assert rv[i] == np.mean([per[i * k + s][2] for s in range(k)])
